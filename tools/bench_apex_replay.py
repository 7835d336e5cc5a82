"""The Ape-X learner iteration of train_apex.py:82-155 with the replay on the host vs on the device.

  (a) host:   Memory (object storage + drl_per_* tree) -> np.stack of the minibatch -> stage + step -> 32 Memory.update
  (b) device: NativeApexReplay.step (sample + gather + step + priority update, one enqueue), then the same loop as K
              back-to-back step_async calls with one wait at the end

Both replays are filled past the wrap with seeded synthetic transitions (a pinned pool reused across adds); ingest is
timed per record of `batch` transitions for both.  target_to_main runs every 100 iterations, as in the reference.
Per-kernel times of the replay kernels come from torch.profiler over a few eager steps.  Prints one JSON line.

    python tools/bench_apex_replay.py [--batch 32] [--capacity 100000] [--iters 300]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FIELDS = ("state", "next_state", "previous_action", "action", "reward", "done")


def _pool(n, A, seed):
    import torch
    rng = np.random.default_rng(seed)

    def pinned(shape, dtype):
        t = torch.empty(shape, dtype={np.uint8: torch.uint8, np.int32: torch.int32, np.float32: torch.float32}[dtype],
                        pin_memory=True)
        return t.numpy()
    p = {"state": pinned((n, 84, 84, 4), np.uint8), "next_state": pinned((n, 84, 84, 4), np.uint8),
         "previous_action": pinned((n,), np.int32), "action": pinned((n,), np.int32),
         "reward": pinned((n,), np.float32), "done": pinned((n,), np.uint8)}
    p["state"][:] = rng.integers(0, 256, p["state"].shape, dtype=np.uint8)
    p["next_state"][:] = rng.integers(0, 256, p["next_state"].shape, dtype=np.uint8)
    p["previous_action"][:] = rng.integers(0, A, n)
    p["action"][:] = rng.integers(0, A, n)
    p["reward"][:] = rng.standard_normal(n).astype(np.float32)
    p["done"][:] = rng.random(n) < 0.1
    return p


def _learner(B, A, graph):
    from distributed_reinforcement_learning_b200.apex_learner import MAIN, TARGET, NativeApexLearner
    from distributed_reinforcement_learning_b200.model import apex_value
    eng = NativeApexLearner(batch=B, num_action=A, use_cuda_graph=graph)
    eng.set_params(apex_value.init_params(num_action=A), MAIN)
    eng.set_params(apex_value.init_params(num_action=A), TARGET)
    return eng


def _card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:
        power = None
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--actions", type=int, default=4)
    ap.add_argument("--capacity", type=int, default=100000)
    ap.add_argument("--iters", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--graph", type=int, default=1)
    a = ap.parse_args()
    import torch
    from distributed_reinforcement_learning_b200.apex_learner import NativeApexReplay
    from distributed_reinforcement_learning_b200.distributed_queue import buffer_queue
    B, A, cap = a.batch, a.actions, a.capacity
    pool = _pool(3 * B, A, seed=1)
    chunk = [{k: pool[k][j * B:(j + 1) * B] for k in FIELDS} for j in range(3)]
    fill = cap + 2 * B
    res = dict(batch=B, num_action=A, capacity=cap, iters=a.iters, use_cuda_graph=bool(a.graph))

    # ---- (a) host replay ----------------------------------------------------------------------------------------
    host = _learner(B, A, bool(a.graph))
    mem = buffer_queue.Memory(cap)

    def host_ingest(rec):
        td = host.td_error(*[rec[k] for k in FIELDS])
        for i in range(len(td)):
            mem.add(td[i], [rec["state"][i], rec["next_state"][i], rec["previous_action"][i], rec["action"][i],
                            rec["reward"][i], rec["done"][i]])

    t0 = time.perf_counter()
    for j in range(fill // B):
        host_ingest(chunk[j % 3])
    res["host_ingest_ms_per_record"] = (time.perf_counter() - t0) * 1e3 / (fill // B)

    def host_iter(it):
        minibatch, idxs, w = mem.sample(B)
        mb = np.array(minibatch, dtype=object)
        slot = it % 2
        host.stage(slot, np.stack(mb[:, 0]), np.stack(mb[:, 1]), np.stack(mb[:, 2]), np.stack(mb[:, 3]),
                   np.stack(mb[:, 4]), np.stack(mb[:, 5]), w)
        _, td = host.step(slot)
        if it % 100 == 0:
            host.target_to_main()
        for i in range(B):
            mem.update(idxs[i], td[i])

    for it in range(a.warmup):
        host_iter(it)
    t0 = time.perf_counter()
    for it in range(a.iters):
        host_iter(it)
    res["host_ms_per_iter"] = (time.perf_counter() - t0) * 1e3 / a.iters
    mem.tree.close()
    host.close()

    # ---- (b) device replay --------------------------------------------------------------------------------------
    dev = _learner(B, A, bool(a.graph))
    rep = NativeApexReplay(dev, cap, seed=2)
    t0 = time.perf_counter()
    for j in range(fill // B):
        rep.add(*[chunk[j % 3][k] for k in FIELDS])
    res["device_ingest_ms_per_record"] = (time.perf_counter() - t0) * 1e3 / (fill // B)

    def dev_iter(it):
        _, td = rep.step(it % 2)
        if it % 100 == 0:
            dev.target_to_main()
        return td

    for it in range(a.warmup):
        dev_iter(it)
    t0 = time.perf_counter()
    for it in range(a.iters):
        dev_iter(it)
    res["device_ms_per_iter"] = (time.perf_counter() - t0) * 1e3 / a.iters
    t0 = time.perf_counter()
    for it in range(a.iters):
        rep.step_async(it % 2)
    dev.wait()
    res["device_async_ms_per_iter"] = (time.perf_counter() - t0) * 1e3 / a.iters
    for k in ("host", "device", "device_async"):
        res[k + "_transitions_per_s"] = B * 1e3 / res[k + "_ms_per_iter"]
    res["ingest_speedup"] = res["host_ingest_ms_per_record"] / res["device_ingest_ms_per_record"]
    res["iter_speedup"] = res["host_ms_per_iter"] / res["device_ms_per_iter"]
    rep.close()
    dev.close()

    # ---- per-kernel device times (eager steps under the profiler) -----------------------------------------------
    eager = _learner(B, A, False)
    rep = NativeApexReplay(eager, 4 * B, seed=3)
    for j in range(4):
        rep.add(*[chunk[j % 3][k] for k in FIELDS])
    rep.step(0)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for it in range(10):
            rep.step(it % 2)
        torch.cuda.synchronize()
    want = {"replay_sample_kernel": "sample_us", "replay_gather_kernel": "gather_us",
            "ordered_update_kernel": "priority_update_us"}
    times = {v: [] for v in want.values()}
    for ev in prof.events():
        for k, v in want.items():
            if k in ev.name and ev.device_type.name == "CUDA":
                times[v].append(float(ev.time_range.elapsed_us()))
    res["kernels"] = {k: (float(np.median(v)) if v else None) for k, v in times.items()}
    rep.close()
    eager.close()
    res["gpu"], res["power_limit_w"] = _card()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
