"""CPU (no GPU needed): the NumPy model of the device replay (oracle/replay_np.py) -- its Philox4x32-10 draws against the
Random123 known answers, and the ordered per-node fold of the leaf-update kernel against sequential SumTree updates --
and the replay entry points failing loudly without a device."""
import ctypes as C

import numpy as np
import pytest

from oracle.per_np import MemoryNP, SumTreeNP
from oracle.replay_np import level_fold, ordered_fold, philox4x32_10, u01


@pytest.mark.parametrize("counter,key,expect", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(counter, key, expect):
    got = tuple(int(v) for v in philox4x32_10(counter, key))
    assert got == expect, ["%08x" % v for v in got]


def test_u01_mapping():
    seed, call, n = 0x123456789ABCDEF0, (1 << 32) + 7, 40
    u = u01(seed, n, call)
    assert u.dtype == np.float64 and u.shape == (n,) and np.all(u >= 0) and np.all(u < 1)
    for i in (0, 5, 39):
        x0, x1, _, _ = [int(v) for v in philox4x32_10((i, call & 0xFFFFFFFF, call >> 32, 0),
                                                      (seed & 0xFFFFFFFF, seed >> 32))]
        bits = ((x0 << 32) | x1) >> 11
        assert u[i] == bits / 2.0 ** 53 and bits < 2 ** 53
    assert not np.array_equal(u01(seed, n, call), u01(seed, n, call + 1))
    assert not np.array_equal(u01(seed, n, call), u01(seed + 1, n, call))
    assert np.array_equal(u01(seed, 8, call), u[:8])           # stratum i's draw does not depend on n


def _random_tree(rng, cap, fill):
    t = SumTreeNP(cap)
    for _ in range(fill):
        t.add((rng.random() * 3 + 0.001) ** 0.6)
    return t


def _sequential(t, leaves, prios):
    for lf, p in zip(leaves, prios):
        t.set_leaf(int(lf), np.float64(p))
    return t.nodes


def _case(rng, cap, B):
    t = _random_tree(rng, cap, int(rng.integers(1, 2 * cap)))
    leaves = rng.integers(cap - 1, 2 * cap - 1, B)
    if B > 2:                                               # forced duplicates, adjacent and far apart
        k = int(rng.integers(1, B))
        leaves[k] = leaves[k - 1]
        leaves[-1] = leaves[0]
    prios = (rng.random(B) * 5 + 0.001) ** 0.6
    return t, leaves, prios


def test_ordered_fold_equals_sequential_updates():
    rng = np.random.default_rng(7)
    caps = [2, 3, 5, 7, 50, 100, 1000, 3000, 2047, 2048]     # non-powers of two, and both sides of one
    for n_case in range(120):
        cap = caps[n_case % len(caps)] if n_case < len(caps) else int(rng.integers(2, 3001))
        B = int(rng.integers(1, 257))
        t, leaves, prios = _case(rng, cap, B)
        before = t.nodes.copy()
        want = _sequential(t, leaves, prios)
        got = ordered_fold(before, leaves, prios)
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), (cap, B)


def test_ordered_fold_of_an_add_batch_with_wrap():
    """An add of n transitions at the cursor: leaves cap-1 + (write + i) % cap, here wrapping twice (n > cap)."""
    rng = np.random.default_rng(3)
    cap, write, n = 13, 9, 32
    t = _random_tree(rng, cap, 20)
    leaves = cap - 1 + (write + np.arange(n)) % cap
    prios = (rng.random(n) + 0.001) ** 0.6
    before = t.nodes.copy()
    assert np.array_equal(ordered_fold(before, leaves, prios), _sequential(t, leaves, prios))


def test_level_synchronous_passes_differ():
    """Why the kernel folds per node: with the leaves at two depths (capacity not a power of two) level-by-level passes
    reorder the adds into some node, and the rounding changes."""
    rng = np.random.default_rng(11)
    differ = 0
    for _ in range(200):
        cap = int(rng.integers(3, 3000))
        if cap & (cap - 1) == 0:
            continue
        t, leaves, prios = _case(rng, cap, int(rng.integers(8, 256)))
        before = t.nodes.copy()
        want = _sequential(t, leaves, prios)
        assert np.array_equal(ordered_fold(before, leaves, prios), want)
        differ += not np.array_equal(level_fold(before, leaves, prios), want)
    assert differ > 0


def test_sampling_model_uses_the_draws():
    """MemoryNP.sample fed with u01(seed, n, call) lands every draw in its stratum's mass."""
    rng = np.random.default_rng(5)
    m = MemoryNP(37)
    for _ in range(50):
        m.add(rng.random())
    n = 8
    u = u01(42, n, 0)
    idx, data, prio, w = m.sample(n, u)
    seg = m.tree.total() / n
    for i in range(n):
        s = seg * i + (seg * (i + 1) - seg * i) * u[i]
        assert seg * i <= s <= seg * (i + 1)
        assert idx[i] == m.tree.find(s) and data[i] == idx[i] - 36 and prio[i] > 0
    assert w.max() == 1.0 and m.beta == pytest.approx(0.401)


def test_replay_entry_points_fail_loudly_without_a_device(native):
    if native.device_count() > 0:
        pytest.skip("a CUDA device is present")
    out = C.c_void_p()
    assert native.lib.drl_apex_replay_create(None, 50, C.c_uint64(0), C.byref(out)) == native.DRL_ERR_CUDA
    assert b"no CPU fallback" in native.lib.drl_last_error()
    assert not out.value
    # there is no replay to act on: the other entry points refuse the null handle instead of crashing
    assert native.lib.drl_apex_replay_step_async(None, 0) == native.DRL_ERR_INVALID
    assert native.lib.drl_apex_replay_add(None, 1, None, None, None, None, None, None) == native.DRL_ERR_INVALID
    assert native.lib.drl_apex_replay_destroy(None) == native.DRL_OK
