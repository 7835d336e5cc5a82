"""NumPy restatement of the device replay's arithmetic (csrc/replay.cu) -- TEST INFRASTRUCTURE ONLY.

* ``philox4x32_10`` / ``u01``: the counter-based draws of the sampling kernel.  Philox4x32-10 with the Random123
  constants; stratum i of draw call c uses counter (i, c lo, c hi, 0) and key (seed lo, seed hi), and
  u = ((x0 << 32 | x1) >> 11) * 2**-53.  Pinned by the Random123 known-answer vectors (tests/test_replay_model.py).
* ``ordered_fold``: the ordered leaf update of ``ordered_update_kernel`` -- change_i = p_i - (leaf value at time i), then
  every touched internal node adds the changes of the updates whose path passes through it, in increasing i.  Equal bit
  for bit to ``SumTreeNP.set_leaf`` applied in order.
* ``level_fold``: the level-synchronous alternative (pass k adds every update's change to its k-th ancestor), which is
  NOT equal when the leaves sit at two depths; kept as the guard of that design note.
* ``ReplayNP``: ``MemoryNP`` driven by those draws, i.e. what the device replay computes given its leaf values.
"""
import numpy as np

from oracle.per_np import MemoryNP

_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_MASK = 0xFFFFFFFF


def philox4x32_10(counter, key):
    """counter: 4 uint32 (scalars or equal-shape arrays), key: 2 uint32 -> 4 uint32 arrays."""
    x = [np.asarray(c, np.uint64) & _MASK for c in counter]
    k0, k1 = [np.asarray(k, np.uint64) & _MASK for k in key]
    for r in range(10):
        if r:
            k0 = (k0 + _W0) & _MASK
            k1 = (k1 + _W1) & _MASK
        p0 = np.uint64(_M0) * x[0]
        p1 = np.uint64(_M1) * x[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & _MASK
        x = [hi1 ^ x[1] ^ k0, lo1, hi0 ^ x[3] ^ k1, lo0]
    return [v.astype(np.uint64) for v in x]


def u01(seed, n, call):
    """[n] float64 uniforms in [0, 1) of draw call `call` for strata 0..n-1."""
    i = np.arange(n, dtype=np.uint64)
    c = int(call)
    x0, x1, _, _ = philox4x32_10((i, c & _MASK, (c >> 32) & _MASK, 0), (int(seed) & _MASK, (int(seed) >> 32) & _MASK))
    bits = ((x0 << np.uint64(32)) | x1) >> np.uint64(11)
    return bits.astype(np.float64) * 2.0 ** -53


def _ancestors(node):
    out = []
    while node != 0:
        node = (node - 1) // 2
        out.append(node)
    return out


def ordered_fold(nodes, leaves, prios):
    """The device's ordered update on a copy of `nodes` (float64 [2 cap - 1]) -> new nodes."""
    t = np.array(nodes, np.float64, copy=True)
    leaves = [int(x) for x in leaves]
    prios = [np.float64(p) for p in prios]
    change = []
    for i, (lf, p) in enumerate(zip(leaves, prios)):
        old = t[lf]
        for j in range(i - 1, -1, -1):
            if leaves[j] == lf:
                old = prios[j]
                break
        change.append(p - old)
    for lf, p in zip(leaves, prios):
        t[lf] = p                                       # the last duplicate wins
    touched = {}
    for i, lf in enumerate(leaves):
        for a in _ancestors(lf):
            touched.setdefault(a, []).append(i)
    for a, js in touched.items():
        acc = nodes[a]
        for j in js:                                    # increasing i
            acc = acc + change[j]
        t[a] = acc
    return t


def level_fold(nodes, leaves, prios):
    """Level-synchronous passes: the changes of every update, one tree level at a time from the deepest up, each level
    in call order.  Differs from the sequential tree when the leaves sit at two depths."""
    t = np.array(nodes, np.float64, copy=True)
    cur = [int(x) for x in leaves]
    change = []
    for i, (lf, p) in enumerate(zip(cur, prios)):
        old = t[lf]
        for j in range(i - 1, -1, -1):
            if cur[j] == lf:
                old = np.float64(prios[j])
                break
        change.append(np.float64(p) - old)
    for lf, p in zip(cur, prios):
        t[lf] = p
    while any(c != 0 for c in cur):            # pass k adds every update's change to its k-th ancestor
        for i, c in enumerate(cur):
            if c != 0:
                cur[i] = (c - 1) // 2
                t[cur[i]] += change[i]
    return t


class ReplayNP:
    """MemoryNP with the device's draws: ``sample`` uses u01(seed, n, call) and advances the call counter."""

    def __init__(self, capacity, seed=0):
        self.mem = MemoryNP(capacity)
        self.seed = int(seed)
        self.calls = 0

    def sample(self, n):
        out = self.mem.sample(n, u01(self.seed, n, self.calls))
        self.calls += 1
        return out
