#!/usr/bin/env python
"""bench.py -- IMPALA learner env-frames/sec on synthetic (T=20, B=32/GPU, 84x84x4) trajectories.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--scaling weak|strong]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one learner update (forward over B*T rows, V-trace, losses, backward, global-norm clip,
TF1-RMSProp) on a batch of B=32 trajectories per GPU (BASELINE.json configs[1]); weak scaling: every rank
holds its own 32 trajectories and the gradient bucket is all-reduced (SUM, NCCL) before the update.

  value  : frames/s with the batch already resident in device staging slots (two slots with different
           data, alternated; the per-step working set, ~230 MB, exceeds the 126 MB L2).
  e2e    : frames/s through the C-ABI with HOST buffers: every step cudaMemcpyAsync's that step's
           19.4 MB batch from the pinned trajectory ring and reads the step's 4 result scalars back.
  roofline / roofline_vtrace : dominant kernel (tensor/FMA bound) and the stand-alone V-trace kernel (HBM).
  cpu_baseline : the CPU oracle (oracle/impala_torch.py, float32, reference-shaped graph: 54 network
           copies, host float64 /255) timed on this box's host cores -- a torch restatement, not TF1.
--impl reference runs only that CPU restatement with the same metric/config (TF 1.14 is not installable).
--batch 4 is BASELINE configs[0] (the reference's own CPU-runnable case) for either arm; --scaling strong shards a
fixed global batch of 256 trajectories over the N GPUs (configs[2]; the default, weak, keeps 32 per GPU).
At N > 1 the line also carries "replicas_identical" (bitwise-equal parameters on every rank after the timed loops) and
"reduce_matches_nccl" (the fused peer exchange's reduced bucket against an NCCL all-reduce of the saved local buckets).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (it may be read-only)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T, A, L, B_PER_GPU = 20, 18, 256, 32
STRONG_GLOBAL_BATCH = 256
METRIC = "learner env-frames/sec (T=20,B=32/GPU,84x84x4)"


def batch_per_gpu(args, world):
    if args.scaling == "strong":
        if STRONG_GLOBAL_BATCH % world:
            raise SystemExit("--scaling strong: %d GPUs do not divide the global batch of %d" % (world, STRONG_GLOBAL_BATCH))
        return STRONG_GLOBAL_BATCH // world
    return args.batch


def bench_config(args, world):
    """The `config` object of BOTH arms (identical by construction: the driver compares them)."""
    B = batch_per_gpu(args, world)
    which = ("BASELINE configs[0]" if (B == 4 and world == 1) else "BASELINE configs[1]" if (B == 32 and world == 1)
             else "BASELINE configs[2]" if world * B == 256 else "BASELINE configs[1] shape")
    return {"workload": "IMPALA learner step (%s): B=%d trajectories/GPU, T=20, 84x84x4 uint8, A=18, LSTM 256; "
                        "glorot random-init parameters" % (which, B),
            "global_batch": world * B, "trajectory": T, "parallelism": "dp%d" % world,
            "scaling_mode": args.scaling,
            "l2": "inputs+activations+params ~%d MB/step %s 126 MB L2; two staging slots alternate"
                  % (int(7.2 * B), ">" if 7.2 * B > 126 else "<"),
            "arms": "ours: hand-written sm_100a kernels behind the C-ABI (csrc/libdrl_b200.so); reference: float32 "
                    "torch-CPU restatement of the TF1 graph on the host cores (TF 1.14 is not installable), a bounded "
                    "sample of min(global_batch, 32) trajectories per step"}


MATH_MODES = {1: "FP32 FFMA (CUDA cores)",
              2: "tcgen05 kind::tf32, 3xTF32 split (A_lo*B_hi + A_hi*B_lo + A_hi*B_hi), fp32 TMEM accumulate",
              3: "tcgen05 kind::tf32 3xTF32, persistent warp-specialised kernels (dedicated epilogue warps)",
              4: "tcgen05 kind::tf32 3xTF32 with TMA-fed conv2/conv3 forward (tensor loads of value + tf32-remainder planes)",
              5: "tcgen05 kind::f16 with 16-bit split operands (A_lo*B_hi + A_hi*B_lo + A_hi*B_hi, fp32 TMEM accumulate; "
                 "bf16 hi/lo planes, uint8 frames exact in fp16)"}


def synth_batch(B, seed):
    """Synthetic trajectories of the shapes/dtypes train_impala.py:100-108 feeds (SURVEY.md 8(d))."""
    rng = np.random.default_rng(seed)
    logits = rng.standard_normal((B, T, A)).astype(np.float32)
    e = np.exp(logits - logits.max(-1, keepdims=True))
    reward = rng.standard_normal((B, T)).astype(np.float32)
    reward[rng.random((B, T)) < 0.1] = 0.0
    return dict(
        state=rng.integers(0, 256, (B, T, 84, 84, 4), dtype=np.uint8),
        reward=reward,
        action=rng.integers(0, A, (B, T)).astype(np.int32),
        done=rng.random((B, T)) < 0.05,
        behavior_policy=(e / e.sum(-1, keepdims=True)).astype(np.float32),
        previous_action=rng.integers(0, A, (B, T)).astype(np.int32),
        initial_h=np.clip(rng.standard_normal((B, T, L)) * 0.5, -0.999, 0.999).astype(np.float32),
        initial_c=rng.standard_normal((B, T, L)).astype(np.float32))


FIELDS = ("state", "reward", "action", "done", "behavior_policy", "previous_action", "initial_h", "initial_c")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


# ---- clocks sampling (B200_PROFILING.md) -------------------------------------------------------
class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region.  The timed region of the default run is
    only tens of milliseconds, shorter than one `nvidia-smi -lms` period, so NVML is polled directly from a
    thread every ~2 ms (same counters as the recipe's nvidia-smi query); nvidia-smi is the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.nvml, self.samples, self.stop_flag, self.th = None, [], False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((mhz, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.th.join(timeout=1)
            if not self.samples:
                return None
            reasons = sorted(k for k, bit in self.BITS.items() if any(rs & bit for _, rs in self.samples))
            return dict(sm_mhz=float(np.median([m for m, _ in self.samples])), sm_max_mhz=self.max_mhz,
                        reasons=reasons, samples=len(self.samples), source="nvml, 2 ms polling")
        if not self.proc:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                 f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                    samples=len(sm), source="nvidia-smi -lms 100")


# ---- FLOP / byte accounting (DESIGN.md section "kernels") ----------------------------------------
def kernel_flops(name, M, Mb):
    tbl = {
        "conv1_fwd": 2.0 * M * 400 * 32 * 256, "conv2_fwd": 2.0 * M * 81 * 64 * 512,
        "conv3_fwd": 2.0 * M * 49 * 64 * 576, "lstm_fwd": 2.0 * M * 1024 * 3648,
        "heads_l1_fwd": 4.0 * M * 256 * 256, "heads_l2_fwd": 4.0 * M * 256 * 256,
        "lstm_wgrad": 2.0 * 3648 * 1024 * Mb, "lstm_dgrad": 2.0 * Mb * 3392 * 1024,
        "conv3_wgrad": 2.0 * Mb * 49 * 64 * 576, "conv3_dgrad": 2.0 * Mb * 49 * 64 * 576,
        "conv2_wgrad": 2.0 * Mb * 81 * 64 * 512, "conv2_dgrad": 2.0 * Mb * 81 * 64 * 512,
        "conv1_wgrad": 2.0 * Mb * 400 * 32 * 256,
        "heads_l2_wgrad": 4.0 * Mb * 256 * 256, "heads_l2_dgrad": 4.0 * Mb * 256 * 256,
        "heads_l1_wgrad": 4.0 * Mb * 256 * 256, "heads_l1_dgrad": 4.0 * Mb * 256 * 256,
    }
    return tbl.get(name)


# DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) per launch at B=32, T=20 from the ncu --set full
# capture summarised in profiles/r01_ncu_umma_full.md (tcgen05 path; conv*_dgrad = the dCol GEMM part only).
NCU_TRAFFIC_B32 = {"lstm_fwd": 38.70e6, "lstm_wgrad": 10.25e6, "lstm_dgrad": 37.94e6, "conv1_fwd": 18.18e6,
                   "conv2_fwd": 33.09e6, "conv3_fwd": 13.62e6, "conv1_wgrad": 46.14e6, "conv2_wgrad": 41.79e6,
                   "conv3_wgrad": 19.22e6, "conv2_dgrad": 49.42e6, "conv3_dgrad": 16.57e6}


# the same for the split-16 kernels (math mode 5), from profiles/r02_ncu_umma16_full.md
# (+ profiles/r02_ncu_conv1_tma.md for the two frame-resident conv1 kernels; lstm_wgrad is the bulk-fed kernel now: not captured)
NCU_TRAFFIC_B32_M5 = {"conv2_fwd": 32.95e6, "conv3_fwd": 13.47e6, "lstm_fwd": 23.68e6,
                      "lstm_dgrad": 23.78e6, "conv3_wgrad": 19.21e6, "conv3_dgrad": 16.60e6, "conv2_wgrad": 41.74e6,
                      "conv2_dgrad": 50.96e6, "conv1_fwd": 18.21e6, "conv1_wgrad": 46.13e6}


def step_flops(B):
    M, Mb = B * T, B * (T - 2)
    return 2.0 * 11810048 * M + 2.0 * 2.0 * 11810048 * Mb       # SURVEY.md App. B (upper bound incl. conv1 dgrad)


# ---- CPU restatement of the reference (oracle) ---------------------------------------------------
def usable_cores():
    """Host cores this process may really use: min(affinity, cgroup CPU quota).  The gpurun boxes show 128
    logical CPUs but carry a 16-CPU cgroup quota; 128 torch threads under that quota run 500x slower
    (profiles/r01_cpu_threads_probe.txt), so the quota is what "all the host threads it can use" means."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def cpu_reference(steps, warmup, B=B_PER_GPU, global_batch=None, budget_s=10.0):
    import torch
    from oracle import impala_torch as it
    from oracle import synthetic
    cores = usable_cores()
    torch.set_num_threads(cores)
    batch = synthetic.make_batch(B, T=T, A=A)
    args = [batch[k] for k in synthetic.TRAIN_FIELDS]
    Lr = it.Learner(None, torch.float32, "reference")
    for _ in range(warmup):
        Lr.train(*args)
    ts = []
    # steps = None: a time-bounded sample (the cpu_baseline leg of the default run): at least 3 steps, then as many as
    # fit into ~10 s of CPU work (task section 4: "about 10-30 s of CPU work"), at most 64
    while (len(ts) < steps) if steps is not None else (len(ts) < 3 or (sum(ts) < budget_s and len(ts) < 64)):
        t0 = time.perf_counter()
        Lr.train(*args)
        ts.append(time.perf_counter() - t0)
    steps = len(ts)
    sec = float(np.sum(ts)) / max(len(ts), 1)
    return dict(value=B * T / sec, unit="frames/s", cores=cores, kind="port", ms_per_step=sec * 1e3,
                sample="%d timed steps (+%d warm-up) of the float32 torch-CPU restatement of the reference graph "
                       "(54 per-timestep network copies, host float64 /255, 2 serial V-trace scans, autograd, "
                       "clip 40, TF1-RMSProp) at B=%d,T=%d%s" % (steps, warmup, B, T,
                       "" if not global_batch or global_batch == B else
                       " (a bounded sample: %d of the workload's %d trajectories per step)" % (B, global_batch)))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    # same steps / warm-up as asked (the CPU step takes ~0.25 s at B=32: K=20, W=5 is ~6 s); a cap keeps an
    # accidental --steps 1000 within a few minutes
    steps, warm = max(1, min(args.steps, 200)), max(1, min(args.warmup, 20))
    cfg = bench_config(args, world)
    B = min(cfg["global_batch"], 32)
    cb = cpu_reference(steps, warm, B, cfg["global_batch"])
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "frames/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg, "cpu_baseline": cb, "gpu_launches": 0,
            "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---- our arm ----------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from distributed_reinforcement_learning_b200.distributed_queue import buffer_queue
    from distributed_reinforcement_learning_b200.learner import NativeLearner
    from distributed_reinforcement_learning_b200.model import impala_actor_critic as model

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    saved_stdout = None
    if world > 1:
        # libraries write to fd 1 behind Python's back (NCCL prints "NCCL version ..." there when the image sets
        # NCCL_DEBUG=VERSION): keep stdout for the ONE JSON line by pointing fd 1 at stderr until that line is printed
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    B, K, W = batch_per_gpu(args, world), args.steps, max(args.warmup, 3)
    M, Mb = B * T, B * (T - 2)
    # N = 1: the whole step is one CUDA graph.  N > 1, --collective peer (default): still one graph, the gradient
    # exchange runs as kernels over NVLink peer memory (csrc/peer.cu); --collective nccl: forward+backward and
    # clip+RMSProp are two graphs with torch.distributed's NCCL all_reduce of the bucket between them.
    use_graph = not args.no_graph
    eng = NativeLearner(batch=B, trajectory=T, num_action=A, device=local, num_slots=2, use_cuda_graph=use_graph,
                        math_mode=args.math_mode)
    eng.set_params(model.init_params(seed=0))
    if world > 1 and args.collective == "peer":
        if not eng.enable_peer_exchange():       # some rank could not map a peer: every rank stays on NCCL
            args.collective = "nccl"
    eng._no_collective = world > 1 and args.collective == "none"
    ext = torch.cuda.ExternalStream(eng.stream_ptr(), device="cuda:%d" % local)

    # host data: 3 distinct batches in a pinned trajectory ring (the FIFOQueue replacement)
    q = buffer_queue.FIFOQueue(T, [84, 84, 4], A, 3 * B, B, 1, L)
    hb = []
    for i in range(3):
        bt = synth_batch(B, 1234 + 17 * rank + i)
        for j in range(B):
            q.append_to_queue(0, bt["state"][j], None, bt["reward"][j], bt["done"][j], bt["behavior_policy"][j],
                              bt["action"][j], bt["previous_action"][j], bt["initial_h"][j], bt["initial_c"][j])
    # pop the three batch slots as pinned views (held: the ring is only a pinned allocator here)
    import ctypes as C
    from distributed_reinforcement_learning_b200 import _native as N
    for i in range(3):
        rb = N.RingBatch()
        N.check(N.lib.drl_ring_pop_batch(q._r, C.byref(rb), 1000))
        v = buffer_queue._view
        hb.append((v(rb.state, (B, T, 84, 84, 4), np.uint8), v(rb.reward, (B, T), np.float32),
                   v(rb.action, (B, T), np.int32), v(rb.done, (B, T), np.uint8),
                   v(rb.behavior_policy, (B, T, A), np.float32), v(rb.previous_action, (B, T), np.int32),
                   v(rb.previous_h, (B, T, L), np.float32), v(rb.previous_c, (B, T, L), np.float32)))
    h2d = int(sum(a.nbytes for a in hb[0]))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- device-resident throughput (`value`) ----------------
    eng.stage(0, *hb[0])
    eng.stage(1, *hb[1])
    for i in range(W):
        eng.step_async(i % 2)
    eng.wait()
    # NVML is initialised BEFORE the barrier (nvmlInit costs milliseconds; started after it, rank 0 entered the timed
    # region late and every other rank's first exchange kernel waited for it), then one more untimed step runs after
    # the barrier so that all ranks enter the timed region from the same, synchronised state.
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    barrier()
    eng.step_async(W % 2)
    eng.wait()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(ext)
    for i in range(K):
        eng.step_async((W + 1 + i) % 2)
    e1.record(ext)
    out = eng.wait()
    barrier()
    ms_dev = max_over_ranks(e0.elapsed_time(e1))
    launches = eng.launches_per_step() * K
    if args.dump_outputs and rank == 0:
        # read back now: the e2e and profiling steps below update the parameters again
        dump_outputs(args.dump_outputs, out, eng.get_params(), eng.get_grads())

    # ---------------- end to end through host buffers (`e2e`) ----------------
    for i in range(2):       # warm the copy path
        eng.stage(i % 2, *hb[i % 3])
        eng.step(i % 2)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    eng.stage(0, *hb[0])
    e2.record(ext)
    per_slot = world == 1 or args.collective == "peer"     # the NCCL path keeps one result record: depth 1
    for i in range(K):
        eng.step_async(i % 2)
        if i + 1 < K:
            eng.stage((i + 1) % 2, *hb[(i + 1) % 3])     # H2D of step i+1 overlaps compute of step i
        if per_slot:
            if i >= 1:
                out = eng.wait((i - 1) % 2)               # D2H read of step i-1's scalars while step i runs
        else:
            out = eng.wait()                              # D2H read of this step's scalars
    if per_slot:
        out = eng.wait((K - 1) % 2)
    e3.record(ext)
    barrier()
    wall_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    ms_e2e = max(max_over_ranks(e2.elapsed_time(e3)), 0.0)
    ms_e2e = max(ms_e2e, wall_ms * 0.0)                   # event time is the reported one; wall kept for reference
    # the sampler covered both timed regions (device-resident and e2e: the same steps, back to back): an NVML query can
    # take milliseconds on a busy GPU, and the first region alone is only K x 0.47 ms long
    clocks = sampler.stop() if sampler else None
    if clocks:
        clocks["window"] = "device-resident + e2e timed regions"

    # ---------------- N > 1: replicas identical? fused exchange == NCCL all-reduce of the local buckets? ----------
    checks = {}
    if world > 1:
        checks = multi_gpu_checks(torch, dist, eng, hb, args, rank, world)

    # ---------------- per-kernel profile -> roofline of the dominant kernel ----------------
    line_extra = dict(checks)
    if rank == 0:
        peaks = measured_peaks()
        eng.stage(0, *hb[0])
        prof = None
        profs = [eng.profile_step(0) for _ in range(3)]
        prof = profs[-1]
        tot = sum(ms for _, ms in prof)
        top = sorted(prof, key=lambda kv: -kv[1])
        # the dominant contraction kernel (the col2im / elementwise sections carry no flop count)
        name, kms = next(((n, ms) for n, ms in top if kernel_flops(n, M, Mb)), top[0])
        fl = kernel_flops(name, M, Mb)
        if fl:
            ach = fl / (kms * 1e-3) / 1e12
            line_extra["roofline"] = {
                "kernel": name, "bound": "tensor", "achieved": ach, "peak": peaks["tf_sus"], "unit": "TFLOP/s",
                "frac": ach / peaks["tf_sus"],
                # fp32-grade results cost 3 tf32 MMAs per product and tf32 runs at half the bf16 rate:
                "frac_of_3xtf32_ceiling": ach / (peaks["tf_sus"] / 6.0) if args.math_mode in (2, 3, 4) else None,
                "frac_of_3x16bit_ceiling": ach / (peaks["tf_sus"] / 3.0) if args.math_mode == 5 else None,
                "traffic": (NCU_TRAFFIC_B32.get(name) if args.math_mode == 2 else
                            NCU_TRAFFIC_B32_M5.get(name) if args.math_mode == 5 else None) if B == 32 else None,
                "traffic_source": (("profiles/r02_ncu_conv1_tma.md" if name.startswith("conv1") else
                                    "profiles/r02_ncu_umma16_full.md") if args.math_mode == 5 else
                                   "profiles/r01_ncu_umma_full.md") + " (ncu --set full, dram read + write per launch)",
                "peak_source": peaks["src"] + " bf16 sustained",
                "math_mode": MATH_MODES[args.math_mode] + "; achieved = algorithmic 2MNK flops (counted once, "
                             "not x3) / CUDA-event time",
                "kernel_ms": kms, "share_of_step": kms / tot}
        line_extra["kernels_ms"] = [[n, round(ms, 4)] for n, ms in top]
        line_extra["step_ms_sum_of_kernels"] = tot
        line_extra["step_tflops"] = step_flops(B) / (ms_dev / K * 1e-3) / 1e12
        # stand-alone V-trace kernel, bandwidth-meaningful size (HBM bound)
        try:
            line_extra["roofline_vtrace"] = vtrace_roofline(torch, peaks)
        except Exception as ex:      # pragma: no cover
            line_extra["roofline_vtrace"] = {"error": str(ex)}
        try:
            line_extra["roofline_vtrace_b32"] = vtrace_roofline(torch, peaks, Bv=32, reps=200)
        except Exception as ex:      # pragma: no cover
            line_extra["roofline_vtrace_b32"] = {"error": str(ex)}
        if args.cpu_baseline and world == 1:      # rank 0 at N=1 only
            line_extra["cpu_baseline"] = cpu_reference(None, 1, min(B, 32), B)
    if world > 1:
        dist.barrier()           # peers' buffers stay mapped until everybody is done
    eng.close()
    if rank == 0 and world == 1 and args.agent_api:
        try:
            line_extra["e2e_agent_api"] = agent_api_e2e(B, K, W, hb, args)
        except Exception as ex:      # pragma: no cover
            line_extra["e2e_agent_api"] = {"error": str(ex)}
    if rank == 0:
        fps = world * B * T / (ms_dev / K * 1e-3)
        fps_e2e = world * B * T / (ms_e2e / K * 1e-3)
        cfg = bench_config(args, world)
        line = {"metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": cfg,
                "impl_detail": {
                    "collective": (None if world == 1 else
                                   "fused reduce-scatter/all-gather kernels over NVLink peer memory (CUDA IPC) "
                                   "inside the step graph" if args.collective == "peer" else
                                   "NCCL all_reduce(SUM) of the 16.6 MB bucket between two graphs"
                                   if args.collective == "nccl" else "NONE (diagnostic, invalid)"),
                    "cuda_graph": bool(use_graph), "math_mode": MATH_MODES[args.math_mode]},
                "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 32,
                        "ms_per_step": ms_e2e / K, "wall_ms_per_step": wall_ms / K,
                        "path": "pinned ring -> drl_learner_stage (copy stream) -> drl_learner_step_async -> "
                                "drl_learner_wait_slot (every step's scalars are read on the host, one step behind: "
                                "two steps in flight), double-buffered slots"},
                "gpu_launches": launches, "clocks": clocks,
                "last_step": {k: out[k] for k in ("pi_loss", "baseline_loss", "entropy", "grad_norm", "step")}}
        line.update(line_extra)
        if saved_stdout is not None:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(d, out, params, grads):
    """What the last timed step returned to its caller: its scalars, the updated parameters and the gradient bucket
    the update consumed (flat, float32, 16.6 MB each at the default shape), as <d>/<name>.npy."""
    os.makedirs(d, exist_ok=True)
    arrays = {k: np.float64(out[k]) for k in ("pi_loss", "baseline_loss", "entropy", "learning_rate", "grad_norm",
                                              "total_loss", "step")}
    arrays.update(params=params, grads=grads)
    for k, v in arrays.items():
        np.save(os.path.join(d, k + ".npy"), v)


# dram__bytes_read.sum + dram__bytes_write.sum per launch of vtrace_from_softmax_pipe_kernel at [65536,18,18], from the
# ncu --set full capture summarised in profiles/r02_ncu_vtrace.md
NCU_TRAFFIC_VTRACE = 201.4e6


def vtrace_roofline(torch, peaks, Bv=65536, Tv=18, reps=20):
    """drl_vtrace_from_softmax_dev on [B,18,18] softmaxes.  Algorithmic bytes per (b,t) element: mu 72 + pi 72 +
    action 4 + discount 4 + reward 4 + value 4 read, vs 4 + rho 4 written = 168 B, plus next_values of which the
    kernel reads only the LAST column (4 B per trajectory: optimizer/vtrace.py:62 uses next_values[:, -1] alone).
    198 MB at B=65536 (> L2: HBM-bound); 97 KB at B=32 (the learner's own size: latency-bound, L2-resident)."""
    import ctypes as C
    from distributed_reinforcement_learning_b200 import _native as N
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(0)
    mu = torch.softmax(torch.randn(Bv, Tv, A, device=dev, generator=g), -1).contiguous()
    pi = torch.softmax(torch.randn(Bv, Tv, A, device=dev, generator=g), -1).contiguous()
    act = torch.randint(0, A, (Bv, Tv), device=dev, dtype=torch.int32)
    disc = torch.full((Bv, Tv), 0.99, device=dev)
    rew = torch.randn(Bv, Tv, device=dev, generator=g)
    val = torch.randn(Bv, Tv, device=dev, generator=g)
    nval = torch.randn(Bv, Tv, device=dev, generator=g)
    vs = torch.empty(Bv, Tv, device=dev)
    rho = torch.empty(Bv, Tv, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream()

    def call():
        N.check(N.lib.drl_vtrace_from_softmax_dev(
            C.c_void_p(mu.data_ptr()), C.c_void_p(pi.data_ptr()), C.c_void_p(act.data_ptr()),
            C.c_void_p(disc.data_ptr()), C.c_void_p(rew.data_ptr()), C.c_void_p(val.data_ptr()),
            C.c_void_p(nval.data_ptr()), Bv, Tv, A, 1.0, C.c_void_p(vs.data_ptr()), C.c_void_p(rho.data_ptr()),
            C.c_void_p(st.cuda_stream)))
    for _ in range(3):
        call()
    # The kernel streams 203 MB (> the 126 MB L2) per launch, so back-to-back launches keep missing L2; timing REPS
    # launches between one pair of events keeps the ~5 us event/launch overhead out of a ~40 us kernel.
    # A single flushed launch is timed as well (reported as kernel_ms_single_flushed).
    REPS = reps
    flush.zero_()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(REPS):
        call()
    b.record(st)
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / REPS
    ts = []
    for _ in range(5):
        flush.zero_()                                    # explicit L2 flush before a single timed launch
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        call()
        b.record(st)
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    nbytes = Bv * Tv * (2 * A * 4 + 4 * 4 + 8) + Bv * 4
    ach = nbytes / (ms * 1e-3) / 1e9
    single = float(np.median(ts))
    big = nbytes > (126 << 20)
    return {"kernel": "vtrace_from_softmax_pipe_kernel", "bound": "hbm", "achieved": ach, "peak": peaks["hbm"],
            "unit": "GB/s", "frac": ach / peaks["hbm"],
            "traffic": NCU_TRAFFIC_VTRACE if (big and Bv == 65536) else None, "peak_source": peaks["src"],
            "bytes_per_launch": nbytes, "bytes_per_element": 168, "kernel_ms": ms, "kernel_ms_single_flushed": single,
            "achieved_single_flushed": nbytes / (single * 1e-3) / 1e9,
            "frac_single_flushed": nbytes / (single * 1e-3) / 1e9 / peaks["hbm"],
            "l2": ("%.0f MB streamed per launch > 126 MB L2" % (nbytes / 1e6) if big else
                   "%.0f KB per launch: L2-resident, launch-latency bound (reported for the learner's own size)"
                   % (nbytes / 1e3)) + "; %d back-to-back launches between one event pair; single = one launch after "
                  "an explicit 256 MB L2 flush" % REPS,
            "shape": [Bv, Tv, A]}


def multi_gpu_checks(torch, dist, eng, hb, args, rank, world):
    """(a) parameters bitwise identical on every rank after everything that ran so far; (b) one more step: the bucket
    the update reads (the fused peer exchange's `reduced` buffer) against an NCCL all-reduce(SUM) of the ranks' saved
    LOCAL gradient buckets.  The sums are formed in different orders (rank order here, NCCL's tree/ring there), so (b)
    is checked to 1e-6 of the largest element, not bitwise."""
    import zlib
    dev = torch.device("cuda", eng.device)
    p = eng.get_params()
    crc = zlib.crc32(p.tobytes())
    t = torch.tensor([crc], dtype=torch.int64, device=dev)
    parts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(parts, t)
    crcs = [int(x.item()) for x in parts]
    res = {"replicas_identical": len(set(crcs)) == 1, "replica_param_crc32": crcs[0]}
    if args.collective == "peer":
        eng.stage(0, *hb[0])
        eng.step(0)                                  # forward, backward, fused exchange, update
        torch.cuda.synchronize()
        local = eng.bucket_tensor().clone()          # this rank's own gradient sums (the backward pass left them there)
        reduced = eng.reduced_tensor().clone()
        dist.all_reduce(local, op=dist.ReduceOp.SUM)
        scale = float(local.abs().max().item())
        err = float((local - reduced).abs().max().item()) / max(scale, 1e-30)
        ok = torch.tensor([1 if err <= 1e-6 else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        res.update(reduce_matches_nccl=bool(int(ok.item())), reduce_vs_nccl_max_rel_err=err)
        p2 = eng.get_params()
        t = torch.tensor([zlib.crc32(p2.tobytes())], dtype=torch.int64, device=dev)
        dist.all_gather(parts, t)
        res["replicas_identical"] = res["replicas_identical"] and len(set(int(x.item()) for x in parts)) == 1
    else:
        res["reduce_matches_nccl"] = None            # the exchange IS the NCCL all-reduce in this mode
    return res


def agent_api_e2e(B, K, W, hb, args):
    """The number a train_impala.py user gets: the UNCHANGED learner loop body (train_impala.py:97-108) on the
    reference-named classes -- queue.sample_batch(), np.stack of every field, impala.Agent.train (blocking, returns
    the step's four scalars) -- with actor threads replaced by a pre-filled pinned ring that is topped up outside the
    timed calls.  One step in flight (the reference's train is synchronous)."""
    from distributed_reinforcement_learning_b200.agent import impala
    from distributed_reinforcement_learning_b200.distributed_queue import buffer_queue
    learner = impala.Agent(trajectory=T, input_shape=[84, 84, 4], num_action=A, lstm_hidden_size=L, discount_factor=0.99,
                           start_learning_rate=0.0006, end_learning_rate=0.0, learning_frame=1000000000,
                           baseline_loss_coef=1.0, entropy_coef=0.05, gradient_clip_norm=40.0,
                           reward_clipping="abs_one", model_name="learner", learner_name="learner")
    learner.set_session(None)
    queue = buffer_queue.FIFOQueue(T, [84, 84, 4], A, 4 * B, B, 1, L)

    def fill(i):
        st, rw, ac, dn, mu, pa, h0, c0 = hb[i % 3]
        for j in range(B):
            queue.append_to_queue(0, st[j], None, rw[j], dn[j].view(np.bool_), mu[j], ac[j], pa[j], h0[j], c0[j])
    ts = []
    for i in range(W + K):
        fill(i)
        t0 = time.perf_counter()
        batch = queue.sample_batch()
        pi_loss, baseline_loss, entropy, learning_rate = learner.train(
            state=np.stack(batch.state), reward=np.stack(batch.reward), action=np.stack(batch.action),
            done=np.stack(batch.done), behavior_policy=np.stack(batch.behavior_policy),
            previous_action=np.stack(batch.previous_action), initial_h=np.stack(batch.previous_h),
            initial_c=np.stack(batch.previous_c))
        if i >= W:
            ts.append(time.perf_counter() - t0)
    learner._engine.close()
    queue.close()
    ms = float(np.median(ts)) * 1e3
    return {"value": B * T / (ms * 1e-3), "unit": "frames/s", "ms_per_step": ms, "ms_per_step_mean": float(np.mean(ts)) * 1e3,
            "path": "FIFOQueue.sample_batch (pinned ring views) -> np.stack per field (zero-copy on ring views) -> "
                    "impala.Agent.train -> drl_learner_stage + drl_learner_step (blocking, host wall clock, median of "
                    "%d calls)" % K, "last": [float(pi_loss), float(baseline_loss), float(entropy), float(learning_rate)]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-graph", action="store_true", help="launch kernels directly instead of CUDA graphs")
    ap.add_argument("--math-mode", type=int, default=5, choices=[1, 2, 3, 4, 5],
                    help="1 = FP32 FFMA contractions, 2 = tcgen05 3xTF32, 5 = tcgen05 kind::f16 with 16-bit split operands (default)")
    ap.add_argument("--no-cpu-baseline", dest="cpu_baseline", action="store_false")
    ap.add_argument("--no-agent-api", dest="agent_api", action="store_false",
                    help="skip the e2e_agent_api leg (the unchanged train_impala.py loop body on impala.Agent)")
    ap.add_argument("--batch", type=int, default=B_PER_GPU,
                    help="trajectories per GPU (32 = BASELINE configs[1], the default; 4 = configs[0])")
    ap.add_argument("--scaling", choices=["weak", "strong"], default="weak",
                    help="weak: --batch trajectories per GPU (default); strong: a global batch of 256 sharded over the GPUs")
    ap.add_argument("--collective", choices=["peer", "nccl", "none"], default="peer",
                    help="N > 1: fused peer-memory gradient exchange (default) or NCCL all_reduce; 'none' = no "
                         "exchange at all (diagnostic: N independent replicas, NOT a valid data-parallel step)")
    ap.add_argument("--workload", choices=["impala", "apex", "r2d2", "a3c"], default="impala",
                    help="impala = the headline IMPALA learner step (default); apex = the Ape-X DQN learner step "
                         "(BASELINE configs[3], tools/bench_apex.py); r2d2 = the R2D2 learner step (configs[4], "
                         "tools/bench_r2d2.py)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs (scalars, parameters, gradients) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "impala" or args.impl != "ours"):
        ap.error("--dump-outputs is implemented for --workload impala --impl ours")
    if args.workload != "impala":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        leg = __import__("bench_" + args.workload)
        leg.run(args, sys.modules[__name__])
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
