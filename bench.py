#!/usr/bin/env python
"""bench.py -- micro-steps/sec of the gradient-accumulation train_op (BASELINE.json metric).

A "step" is ONE micro-step of the hot path (one `session.run(train_op)` of the reference,
optimization.py:91-104) on synthetic BERT-Small-shaped gradients: N-1 accumulate launches and one
accumulate+clip+AdamWeightDecay apply launch per window of N.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload bert_small]
                  [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU, NCCL)

`--dump-outputs DIR` writes what the last timed micro-step left for its caller as DIR/<name>.npy
(see dump_outputs); the inputs are seeded, so two builds run with the same arguments can be compared
output for output.

`value`     : whole-job micro-batches/s with gradients already resident in HBM (all ranks).
`e2e`       : same metric through the public host-buffer call: gradients start in pinned host
              memory (H2D every micro-step), updated parameters return to host memory on apply
              steps and the stats block every step (D2H), all inside the timed region.
`roofline`  : the apply kernel's algorithmic 36 B/param over its CUDA-event duration vs the
              measured HBM copy bandwidth in MEASURED_PEAKS.json.
`cpu_baseline`: the CPU oracle (oracle/oracle.c, un-fused op-for-op port of optimization.py, all
              host cores) timed on whole windows of the same workload in the same run.
L2 is defeated by rotating three independent state sets (each > L2) between launches.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

WORKLOADS = {
    # name -> (manifest key, default N, description)   BASELINE.json configs
    "mnist_cnn": ("mnist_cnn", 4, "distributedExample/02 MNIST CNN accum x4 (variant B: tf.train.AdamOptimizer, no clip)"),
    "bert_small": ("bert_small", 4, "BERT-Small L4_H512_A8 seq128 micro_bs8 accum x4"),
    "bert_base": ("bert_base", 8, "BERT-Base L12_H768_A12 seq128 micro_bs32 accum x8"),
    "bert_large": ("bert_large", 32, "BERT-Large L24_H1024_A16 seq512 micro_bs4 accum x32"),
}
INIT_LR, TRAIN_STEPS, WARMUP_STEPS = 2e-5, 207900, 20790      # reference README.md:72,75
START_STEP = 100000      # steady state, mid-schedule (the per-set phases are added in run_b200_arm)
# ONE metric string for both arms: the driver divides the two lines only when they name the same metric
METRIC = "micro-steps/sec (train_op: accumulate + clip_by_global_norm + AdamWeightDecay apply, one window of N = N-1 accumulate + 1 apply)"
PARITY_TOL = 1e-5        # BASELINE.json north_star: "within 1e-5 rel fp32"


def rotation_for(accum_n: int) -> int:
    """Number of rotating state sets: the smallest R >= 3 coprime with N, so that stepping the sets
    round-robin can put exactly one apply launch in every N consecutive bench steps."""
    import math
    r = 3
    while math.gcd(r, accum_n) != 1:
        r += 1
    return r


def set_phase(r: int, R: int, N: int) -> int:
    """global_step offset (mod N) of rotating set r such that, with set (i % R) used at bench step i, the
    apply branch (optimization.py:91: pre-increment step % N == 0) fires exactly at i % N == N-1."""
    if N == 1:
        return 0
    r_inv = pow(R, -1, N)
    j_r = ((-1 - r) * r_inv) % N          # the uses j of set r (bench step r + R*j) that must apply
    return (-j_r) % N


def set_start_step(r: int, R: int, N: int) -> int:
    return START_STEP - START_STEP % N + set_phase(r, R, N)


DUMP_SAMPLE = 1 << 21    # elements kept per dumped array: four 8 MB arrays stay well inside 64 MB at any workload size


def dump_outputs(out_dir, op, params, dp, rank):
    """Writes what the last timed micro-step left for its caller, as float32 DIR/<name>.npy: the updated parameters
    (param), the optimizer state the next micro-step reads (adam_m, adam_v, accum), each flattened in manifest order
    without the slab padding, and the stats block (stats: applied, lr, global_norm, clip_scale).  Arrays longer than
    DUMP_SAMPLE keep the same sorted sample of indices, drawn from a fixed seed.  Under data parallelism every rank
    must call it (the moments are gathered from their shards); rank 0 writes."""
    import numpy as np
    import torch
    state = dp.gather_state() if dp is not None else {"m": op.m, "v": op.v}
    st = op.stats()
    if rank != 0:
        return

    def flat(slab):
        return torch.cat([slab[o:o + p.numel()] for o, p in zip(op.plan.offsets, params)])
    arrays = {"param": torch.cat([p.reshape(-1) for p in params]), "adam_m": flat(state["m"]),
              "adam_v": flat(state["v"]), "accum": flat(op.accum)}
    n = arrays["param"].numel()
    idx = None
    if n > DUMP_SAMPLE:
        idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))).to(op.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), (a if idx is None else a[idx]).cpu().numpy())
    np.save(os.path.join(out_dir, "stats.npy"),
            np.array([st["applied"], st["lr"], st["global_norm"], st["clip_scale"]], dtype=np.float32))


def _finite(x):
    """JSON has no NaN/Infinity: a leg that saw no launch of a kind reports null instead."""
    if isinstance(x, float):
        return x if x == x and abs(x) != float("inf") else None
    if isinstance(x, dict):
        return {k: _finite(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_finite(v) for v in x]
    return x


def manifest(name):
    from gaccum_b200.manifests import MANIFESTS       # the product's own shape tables (never the oracle's)
    return MANIFESTS[WORKLOADS[name][0]]()


def kernel_source_stamp():
    """sha256 over the kernel sources and build flags: ties an ncu traffic capture to the code it measured."""
    import hashlib
    from gaccum_b200 import build as b
    h = hashlib.sha256()
    for name in sorted(b.DEPS):
        with open(os.path.join(b.CSRC, name), "rb") as f:
            h.update(name.encode() + b"\0" + f.read())
    h.update(" ".join(b.NVCC_FLAGS).encode())
    return h.hexdigest()[:16]


def measured_traffic(workload, kernel):
    """dram__bytes_read + dram__bytes_write per launch of the dominant kernel, from the ncu capture
    tools/measure_traffic.py wrote into profiles/traffic.json.  Returned only when the capture was taken
    on this workload, this kernel and THESE kernel sources (stamp); otherwise null, never a stale number."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        e = t["captures"][workload]
        if e["stamp"] != kernel_source_stamp() or e["kernel"] not in kernel:
            return None, f"profiles/traffic.json capture is for other sources/kernel (stamp {e['stamp']})"
        return int(e["dram_bytes"]), f"profiles/traffic.json: ncu dram__bytes_read.sum+dram__bytes_write.sum per launch, stamp {e['stamp']}"
    except Exception:
        return None, "no capture for this workload in profiles/traffic.json"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
# clocks during the timed region (NVML; B200_PROFILING.md "clocks line")
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int, period_s: float = 0.02):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.period = period_s

    def _once(self):
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                     "sw_thermal_slowdown": 0x20, "hw_power_brake": 0x80, "sync_boost": 0x10,
                     "applications_clocks": 0x2}
            for k, bit in names.items():
                if r & bit:
                    self.reasons.add(k)
        except Exception:
            pass

    def start(self):
        if self.nv is None:
            return
        def loop():
            while not self._stop.is_set():
                self._once()
                self._stop.wait(self.period)
        self._thr = threading.Thread(target=loop, daemon=True)
        self._thr.start()

    def stop(self):
        if self._thr is not None:
            self._once()
            self._stop.set()
            self._thr.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "samples": len(s), "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------
# CPU reference leg (oracle/oracle.c on all host cores)
# ------------------------------------------------------------------------------------------------
def cpu_reference(workload: str, accum_n: int, budget_s: float, variant_b: bool):
    """Times whole windows of the un-fused CPU port.  Returns (micro-steps/s, dict)."""
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle_c
    import oracle_np as onp
    man = onp.MANIFESTS[WORKLOADS[workload][0]]()       # the CPU leg stands on the oracle alone
    rng = np.random.default_rng(19830610)
    params = [rng.normal(0, 0.02, s).astype(np.float32) for _, s in man]
    hp = onp.HParams.tf_adam() if variant_b else onp.HParams.bert()
    kw = dict(constant_lr=1e-4) if variant_b else dict(init_lr=INIT_LR, num_train_steps=TRAIN_STEPS, num_warmup_steps=WARMUP_STEPS)
    op = oracle_c.COracleTrainOp(params, [n for n, _ in man], hp, accum_n, global_step=1, **kw)
    grads = [rng.normal(0, 1e-3, s).astype(np.float32) for _, s in man]
    for _ in range(accum_n):                   # one warm-up window (first-touch of scratch)
        op.run(grads)
    # "all the host threads it can use": the un-fused loops are DRAM-bound, and on SMT hosts one thread
    # per logical CPU is slower than one per core -- time one window at each plausible count, keep the best
    ncpu = os.cpu_count() or 1
    best = None
    t_cal = time.perf_counter()
    for nthr in sorted({ncpu, max(1, ncpu // 2), max(1, ncpu // 4)}, reverse=True):
        if best is not None and time.perf_counter() - t_cal > 0.5 * budget_s:
            break                                  # calibration is part of the budget
        oracle_c.set_num_threads(nthr)
        for _ in range(accum_n):
            op.run(grads)
        t0 = time.perf_counter()
        for _ in range(accum_n):
            op.run(grads)
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, nthr)
    oracle_c.set_num_threads(best[1])
    times, t_total = [], 0.0
    while t_total < budget_s and len(times) < 50:
        t0 = time.perf_counter()
        for _ in range(accum_n):
            op.run(grads)
        dt = time.perf_counter() - t0
        times.append(dt); t_total += dt
    times.sort()
    med = times[len(times) // 2]
    rate = accum_n / med
    info = {"value": rate, "unit": "micro-steps/s", "cores": oracle_c.num_threads(), "kind": "port",
            "sample": f"{len(times)} whole windows of {accum_n} micro-steps ({workload}, T={len(man)}), median window {med*1e3:.1f} ms, "
                      f"oracle/oracle.c un-fused OpenMP port of optimization.py (TensorFlow is not installable here)",
            "host_cpus": os.cpu_count()}
    return rate, info, med


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    N = args.accum_n or WORKLOADS[wl][1]
    t0 = time.perf_counter()
    budget = args.cpu_budget if args.cpu_budget_given else min(60.0, 0.05 * max(args.steps, 1) + 10.0)
    rate, info, med = cpu_reference(wl, N, budget_s=budget, variant_b=(wl == "mnist_cnn"))
    import oracle_np
    man = oracle_np.MANIFESTS[WORKLOADS[wl][0]]()
    out = {"impl": "reference", "metric": METRIC, "value": rate,
           "unit": "micro-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1e3 / rate, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{wl}_accum{N}", "T": len(man), "accum_n": N,
                      "note": "steps are bounded: whole windows are timed until the budget is spent; rate is per micro-step"},
           "cpu_baseline": info,
           "e2e": {"value": rate, "unit": "micro-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
    print(json.dumps(_finite(out)))


# ------------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200_arm(args):
    import numpy as np
    import torch
    import gaccum_b200 as g
    from gaccum_b200.train_op import GaccumTrainOp

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    wl = args.workload
    N = args.accum_n or WORKLOADS[wl][1]
    variant_b = wl == "mnist_cnn"
    man = manifest(wl)
    names = [n for n, _ in man]
    K, W = args.steps, max(args.warmup, 3)
    R = rotation_for(N)                             # rotating state sets: defeats the 126 MB L2
    gen = torch.Generator(device=dev); gen.manual_seed(19830610 + 1000 * rank)

    def lr_fn(s):
        return 1e-4 if variant_b else g.learning_rate(INIT_LR, TRAIN_STEPS, WARMUP_STEPS, s)

    NG = min(N, 4)          # distinct gradient sets per state set (BERT-Large x N=32 would not fit otherwise)
    hp = g.HParams.tf_adam() if variant_b else g.HParams.bert()
    if args.no_clip:
        hp.clip_norm = 0.0

    # ---- parity self-check (driver-visible): 2N+1 micro-steps from global_step 0 against the CPU oracle
    #      fed the rank-summed gradients; replicas must be bit-identical.  rc != 0 above 1e-5. ----
    parity = None
    if args.parity_steps != 0:
        parity = parity_check(args, wl, N, hp, variant_b, man, names, world, rank, dev, dist)
        if parity is not None and not parity["ok"]:
            if rank == 0:
                print(json.dumps(_finite({"impl": "b200", "metric": METRIC, "parity": parity,
                                          "error": "parity self-check failed; nothing was timed"})))
            if dist is not None:
                dist.destroy_process_group()
            raise SystemExit(3)

    sets = []
    pgen = torch.Generator(device=dev); pgen.manual_seed(7)        # identical replicas on every rank
    for r in range(R):
        params = [torch.randn(s, device=dev, generator=pgen) * 0.02 for _, s in man]
        dp = None
        # steady state, mid-schedule.  Set (i % R) serves bench step i; its global_step phase is chosen so
        # that the apply branch fires exactly at i % N == N-1: every N consecutive bench steps are one
        # window's launches (N-1 accumulate + 1 apply) while consecutive launches never share a state set.
        gs0 = set_start_step(r, R, N)
        if world > 1 and args.dp == "fused":
            from gaccum_b200.distributed import FusedDataParallelTrainOp
            dp = FusedDataParallelTrainOp(params, names, hp, N, lr_fn, global_step=gs0)
            op = dp.engine
        else:
            op = GaccumTrainOp(params, names, hp, N, lr_fn, global_step=gs0)
        op.m.normal_(0, 1e-4, generator=gen); op.v.uniform_(0, 1e-8, generator=gen)
        grads = [[torch.randn(s, device=dev, generator=gen) * args.sigma for _, s in man] for _ in range(NG)]
        bound = [op.bind(gl) for gl in grads]      # what a graph-mode caller hands the op: raw pointers
        sets.append((op, params, grads, bound, dp))
    P = sets[0][0].plan.num_elements
    stream = torch.cuda.current_stream(dev)

    cuda_stream = stream.cuda_stream

    def micro_step(i):
        op, _, grads, bound, dp = sets[i % R]
        gl = grads[(i // R) % NG]
        if world == 1:
            return op.run_bound(bound[(i // R) % NG], cuda_stream)
        if dp is not None:
            return dp.run_bound(bound[(i // R) % NG], cuda_stream)
        # data parallel (04:55,58 semantics with ONE reduction per window): accumulate locally,
        # all-reduce the packed slab on the apply step only, then apply without a gradient.
        if g.is_apply_step(op.global_step, N):
            op.accumulate_only(gl)
            dist.all_reduce(op.accum)
            op.apply_only(None)
            op.global_step += 1
            return True
        return op.run(gl)

    # warm-up: at least W micro-steps per state set, rounded up to whole windows so that the timed region
    # starts on a window boundary (bench step index % N == 0)
    WU = -(-(W * R) // N) * N
    for i in range(WU):
        micro_step(i)
    # everything slow and rank-dependent (NVML init of the clock sampler, event creation) happens BEFORE the barrier: ranks
    # must enter the timed loop together, or the early ones spend their first exchange waiting for the latest and that
    # wait lands in their timed region (8 GPUs: up to 7 ms of a 32 ms region)
    sampler = ClockSampler(local)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    kinds = []
    sampler.start()
    torch.cuda.synchronize(dev)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(dev)
    base = WU
    torch.cuda.profiler.start()      # ncu --profile-from-start off captures only the timed region
    evs[0].record(stream)
    for i in range(K):
        kinds.append(micro_step(base + i))
        if not args.no_launch_events or i == K - 1:
            evs[i + 1].record(stream)
    torch.cuda.synchronize(dev)
    torch.cuda.profiler.stop()
    clocks = sampler.stop()
    if dist is not None:
        dist.barrier()
    if args.dump_outputs:
        op, params, _, _, dp = sets[(base + K - 1) % R]
        dump_outputs(args.dump_outputs, op, params, dp, rank)
    total_ms = evs[0].elapsed_time(evs[K])
    per = [evs[i].elapsed_time(evs[i + 1]) for i in range(K)] if not args.no_launch_events else [total_ms / K] * K
    if dist is not None:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    apply_ms = [p for p, k in zip(per, kinds) if k]
    acc_ms = [p for p, k in zip(per, kinds) if not k]
    mean = lambda x: (sum(x) / len(x)) if x else float("nan")
    per_rank = None
    if dist is not None:
        # every rank's own per-kind means and total: a straggler (slower GPU, later launches) shows up here, not in rank 0's numbers
        mine = torch.tensor([mean(apply_ms) if apply_ms else 0.0, mean(acc_ms) if acc_ms else 0.0, evs[0].elapsed_time(evs[K])],
                            device=dev, dtype=torch.float64)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank = {"apply_step_us": [round(float(t[0]) * 1e3, 1) for t in allr],
                    "accumulate_us": [round(float(t[1]) * 1e3, 1) for t in allr],
                    "timed_region_ms": [round(float(t[2]), 3) for t in allr]}

    # ---- e2e: the C ABI's host-buffer entry point (gaccum_step_host): parameters and gradients
    #      live in pinned HOST memory; H2D of every micro-step's gradients, D2H of the stats block
    #      every step and of the updated parameters on apply steps are all inside the timed region ----
    e2e = None
    if args.e2e_steps > 0:
        from gaccum_b200.train_op import HostTrainOp
        # allocate (first-touch) the pinned host buffers on the NUMA node next to this GPU, as a
        # NUMA-aware host framework would: bind to the GPU's ideal CPUs while allocating
        old_aff, numa = None, "default placement"
        try:
            import pynvml
            pynvml.nvmlInit()
            old_aff = os.sched_getaffinity(0)
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
            numa = f"pinned buffers first-touched on the GPU-local CPUs ({len(os.sched_getaffinity(0))} of {len(old_aff)})"
        except Exception:
            old_aff = None
        # the caller keeps parameters and gradients in pinned ARENAS laid out like the device slabs (plan offsets):
        # gaccum_step_host then moves each direction with one copy instead of one per tensor
        shapes = [s for _, s in man]
        pflat, host_params = HostTrainOp.pinned_arena(shapes, hp)
        gen_h = torch.Generator(); gen_h.manual_seed(7)             # identical replicas on every rank
        for hp_t in host_params:
            hp_t.copy_(torch.randn(hp_t.shape, generator=gen_h) * 0.02)
        host_grads = []
        for _ in range(2):
            gflat, views = HostTrainOp.pinned_arena(shapes, hp)
            gflat.normal_(0, args.sigma / world)                    # 04:46 loss / num_workers
            host_grads.append(views)
        if old_aff is not None and not args.e2e_keep_affinity:
            os.sched_setaffinity(0, old_aff)
        hop = HostTrainOp(host_params, names, hp, N, lr_fn, global_step=START_STEP - START_STEP % N + 1, device=local)
        if world > 1:
            hop.connect_data_parallel()        # 04:55-62: the apply step becomes the fused NVLink exchange + apply kernel
        hb = [hop.bind(hg) for hg in host_grads]
        Ke = -(-args.e2e_steps // N) * N       # whole windows
        for i in range(N):
            hop.run_bound(hb[i % 2])
        hop.sync()
        if dist is not None:
            dist.barrier()
        napply = 0
        t0 = time.perf_counter()
        for i in range(Ke):
            napply += bool(hop.run_bound(hb[i % 2]))
        hop.sync()
        ms = (time.perf_counter() - t0) * 1e3        # host wall clock around enqueue + sync: the caller's view
        if dist is not None:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        e2e = {"value": world * Ke / (ms * 1e-3), "unit": "micro-steps/s",
               "h2d_bytes_per_step": 4 * P, "d2h_bytes_per_step": int(4 * P * napply / Ke) + 16,
               "steps": Ke, "ms_per_step": ms / Ke, "api": "gaccum_step_host (C ABI) via HostTrainOp.run_bound",
               "host_memory": numa,
               "note": "pinned host gradients H2D every micro-step (one coalesced copy: arena in slab layout); stats D2H every step; "
                       "parameters D2H on apply steps" + ("" if world == 1 else
                       f"; data parallel over {world} ranks: the apply step is the fused NVLink exchange + apply kernel over CUDA-IPC "
                       "peer mappings (gaccum_host_session_dp_connect), accumulate steps are rank-local")}
        del hop

    # ---- with the model in the loop: PyTorch BERT forward/backward (NOT our path) produces the
    #      gradients, then the same train_op; shows what the exchange costs in a real micro-step ----
    with_model = None
    if args.model_steps > 0 and wl in ("bert_small", "bert_base", "bert_large"):
        with_model = with_model_leg(args, wl, N, hp, lr_fn, world, rank, dev, dist)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    # own kernels launched per rank inside the timed region: one per micro-step, plus whatever extra the
    # data-parallel apply step needs (fused: none; nccl all-reduce baseline: accumulate + apply = 2)
    per_apply = getattr(sets[0][4], "launches_per_apply", 2) if world > 1 else 1
    launches_per_rank = K + len(apply_ms) * (per_apply - 1)
    ab = sets[0][0].plan.algorithmic_bytes(True)
    acb = sets[0][0].plan.algorithmic_bytes(False)
    a_ms, c_ms = mean(apply_ms), mean(acc_ms)
    achieved = ab / (a_ms * 1e-3) / 1e9 if apply_ms else float("nan")
    if world == 1:
        kernel = ("apply_clip_kernel (a+=G, /N, global-norm clip, AdamWeightDecay, a=0; one cooperative launch: TMA-fed rings, ticketed tiles, Tensor-Memory stash, exact norm)"
                  if hp.clip_norm > 0 else "apply_kernel (single pass: a+=G, /N, Adam, a=0; no clip)")
    else:
        kernel = "dp_apply_kernel (apply step at N>1: includes the NVLink exchange, so this is not an HBM roofline)"
    traffic, traffic_src = measured_traffic(wl, kernel) if world == 1 else (None, "not captured at N>1")
    window_exact = len(apply_ms) * (N - 1) == len(acc_ms)
    # window-exact rate from the per-kind means (what any whole number of windows costs), beside `value`
    window_us = ((N - 1) * c_ms + a_ms) * 1e3 if (apply_ms and (acc_ms or N == 1)) else None
    out = {
        "impl": "b200",
        "metric": METRIC,
        "value": world * K / (total_ms * 1e-3), "unit": "micro-steps/s", "n_gpus": world, "steps": K, "warmup": WU,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{wl}_accum{N}", "desc": WORKLOADS[wl][2], "T": len(man), "P": P, "accum_n": N,
                   "optimizer": "tf.train.AdamOptimizer" if variant_b else "AdamWeightDecay+clip_by_global_norm(1.0)",
                   "grad_sigma": args.sigma,
                   "parallelism": f"dp{world}" + ("" if world == 1 else
                                                   " fused apply kernel: local a+=G + reduce-scatter + sharded update + all-gather over NVLink peer memory in one launch"
                                                   if args.dp == "fused" else " nccl all-reduce of the packed accum slab on apply steps"),
                   "l2": f"rotating {R} independent state sets ({R * 5 * 4 * P / 1e6:.0f} MB of state+grads per rotation) > 126 MB L2",
                   "apply_launches": len(apply_ms), "accumulate_launches": len(acc_ms),
                   "window_exact": window_exact,
                   "window_exact_value": (world * N / (window_us * 1e-6)) if window_us else None,
                   "mix_note": "bench step i uses state set i % R and applies iff i % N == N-1 (phased global_steps); "
                               "the timed region starts on a window boundary, so K % N == 0 gives exactly K/N windows"},
        "roofline": {"bound": "hbm", "kernel": kernel,
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "peak_source": peak_src, "algorithmic_bytes": ab, "avg_launch_us": a_ms * 1e3,
                     "traffic": traffic, "traffic_source": traffic_src},
        "roofline_accumulate": {"bound": "hbm", "kernel": "accumulate_kernel", "achieved": acb / (c_ms * 1e-3) / 1e9 if acc_ms else None,
                                "peak": peak, "unit": "GB/s", "frac": (acb / (c_ms * 1e-3) / 1e9 / peak) if acc_ms else None,
                                "algorithmic_bytes": acb, "avg_launch_us": c_ms * 1e3 if acc_ms else None},
        "gpu_launches": launches_per_rank,
        "clocks": clocks,
    }
    if parity is not None:
        out["parity"] = parity
    if per_rank is not None:
        out["per_rank"] = per_rank
    if e2e:
        out["e2e"] = e2e
    if with_model:
        out["with_model"] = with_model
    if world == 1 and args.cpu_budget > 0:
        # The CPU leg runs in a fresh interpreter: in this process PyTorch's bundled OpenMP runtime is
        # already loaded (active spin-waiting, its own thread settings) and starves the oracle's loops.
        import subprocess
        env = dict(os.environ, OMP_WAIT_POLICY="PASSIVE")
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", wl, "--accum-n", str(N),
               "--steps", str(K), "--warmup", str(W), "--cpu-budget", str(args.cpu_budget)]
        try:
            r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=args.cpu_budget * 6 + 120)
            line = [l for l in r.stdout.splitlines() if l.startswith("{")][-1]
            out["cpu_baseline"] = json.loads(line)["cpu_baseline"]
        except Exception as e:       # never lose the GPU line because the CPU leg failed
            out["cpu_baseline"] = {"value": None, "unit": "micro-steps/s", "cores": None, "kind": "port",
                                   "sample": f"CPU leg failed: {type(e).__name__}: {e}"}
    print(json.dumps(_finite(out)))
    if dist is not None:
        dist.destroy_process_group()


def parity_check(args, wl, N, hp, variant_b, man, names, world, rank, dev, dist):
    """Driver-visible parity of the path that is about to be timed (reference semantics:
    optimization.py:76-104 on one GPU; 04_multi_worker_with_estimator_gaccum.py:46,55,58,62 on W GPUs).

    Every rank runs `steps` micro-steps from global_step 0 (so the windows are {0}, {1..N}, {N+1..2N}) on
    the workload's real shapes with gradients from numpy PCG64(19830610 + 1000*rank + step), pre-divided by
    the number of workers as 04:46 does.  Rank 0 feeds the CPU oracle (checker use of oracle/) the
    rank-ordered fp32 sum of all ranks' gradients and compares parameters, adam_m, adam_v after the last
    step; replicas are compared bit for bit through int32 min/max all-reduces of the parameter slab."""
    import numpy as np
    import torch
    import gaccum_b200 as g
    from gaccum_b200.train_op import GaccumTrainOp
    Np = min(N, 4)                                   # parity window (keeps BERT-Large x N=32 affordable)
    steps = args.parity_steps if args.parity_steps > 0 else 2 * Np + 1
    sigma = args.sigma
    if variant_b:
        lr_kw, lr_fn = dict(constant_lr=1e-4), (lambda s: 1e-4)
    else:
        # a short schedule so that lr is O(init_lr) from the first apply on (warm-up of 2 micro-steps)
        sched = dict(init_lr=INIT_LR, num_train_steps=1000, num_warmup_steps=2)
        lr_kw, lr_fn = sched, (lambda s: g.learning_rate(sched["init_lr"], sched["num_train_steps"], sched["num_warmup_steps"], s))
    prng = np.random.Generator(np.random.PCG64(19830610))
    host_params = [prng.standard_normal(s, dtype=np.float32) * np.float32(0.02) for _, s in man]
    params = [torch.from_numpy(p).to(dev) for p in host_params]
    dp = None
    if world > 1 and args.dp == "fused":
        from gaccum_b200.distributed import FusedDataParallelTrainOp
        dp = FusedDataParallelTrainOp(params, names, hp, Np, lr_fn)
        op, runner = dp.engine, dp
    elif world > 1:
        from gaccum_b200.distributed import DataParallelTrainOp
        op = GaccumTrainOp(params, names, hp, Np, lr_fn)
        runner = DataParallelTrainOp(op, None)
    else:
        op = runner = GaccumTrainOp(params, names, hp, Np, lr_fn)
    ref = None
    if rank == 0:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import oracle_c
        import oracle_np as onp
        ohp = onp.HParams.tf_adam() if variant_b else onp.HParams.bert()
        ohp.clip_norm = float(hp.clip_norm)
        ref = oracle_c.COracleTrainOp([p.copy() for p in host_params], names, ohp, Np, **lr_kw)
    sizes = [int(np.prod(s)) for _, s in man]
    Ptot = sum(sizes)
    flat = torch.empty(Ptot, dtype=torch.float32, device=dev)
    gathered = [torch.empty_like(flat) for _ in range(world)] if (world > 1 and rank == 0) else None
    t0 = time.perf_counter()
    for step in range(steps):
        rng = np.random.Generator(np.random.PCG64(19830610 + 1000 * rank + step))
        hg = rng.standard_normal(Ptot, dtype=np.float32) * np.float32(sigma / world)    # 04:46 loss / num_workers
        flat.copy_(torch.from_numpy(hg))
        grads, o = [], 0
        for (_, shp), n in zip(man, sizes):
            grads.append(flat[o:o + n].view(shp)); o += n
        runner.run(grads)
        if world > 1:
            dist.gather(flat, gathered, dst=0)
        if rank == 0:
            if world > 1:
                tot = gathered[0].clone()
                for w in range(1, world):
                    tot += gathered[w]                       # fp32, rank order
                hsum = tot.cpu().numpy()
            else:
                hsum = hg
            og, o = [], 0
            for (_, shp), n in zip(man, sizes):
                og.append(hsum[o:o + n].reshape(shp)); o += n
            ref.run(og)
    torch.cuda.synchronize(dev)
    st = op.stats()
    # replicas: bitwise identity of the parameters on every rank
    identical = True
    if world > 1:
        pslab = dp.param_slab if dp is not None else torch.cat([p.reshape(-1) for p in params])
        lo = pslab.view(torch.int32).clone(); hi = lo.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        identical = bool(torch.equal(lo, hi))
    full = dp.gather_state() if dp is not None else {"m": op.m, "v": op.v}
    out = None
    if rank == 0:
        worst, worst_at = 0.0, None
        offs = op.plan.offsets
        hm, hv = full["m"].cpu().numpy(), full["v"].cpu().numpy()
        for i, (nm, shp) in enumerate(man):
            n = sizes[i]
            for kind, got, exp in (("param", params[i].cpu().numpy(), ref.params[i]),
                                   ("adam_m", hm[offs[i]:offs[i] + n].reshape(shp), ref.m[i]),
                                   ("adam_v", hv[offs[i]:offs[i] + n].reshape(shp), ref.v[i])):
                denom = max(float(np.max(np.abs(exp))) if n else 0.0, 1e-30)
                e = float(np.max(np.abs(got.astype(np.float64) - exp.astype(np.float64)))) / denom if n else 0.0
                if not (e <= worst):                        # NaN-safe: a NaN error becomes the worst
                    worst, worst_at = e, f"{kind}:{nm}"
        ok = bool(worst <= PARITY_TOL) and identical
        out = {"max_rel_err": worst, "worst": worst_at, "tol": PARITY_TOL, "replicas_identical": identical, "world": world,
               "steps": steps, "accum_n": Np, "applies": sum(1 for s_ in range(steps) if s_ % Np == 0),
               "last_clip_scale": st["clip_scale"], "last_global_norm": st["global_norm"],
               "oracle": "oracle/oracle.c (CPU restatement of optimization.py) fed the fp32 rank-ordered sum of all ranks' gradients",
               "grads": "numpy PCG64(19830610 + 1000*rank + step), N(0, sigma^2)/world", "wall_s": time.perf_counter() - t0,
               "ok": ok}
    if world > 1:
        flag = torch.tensor([1 if (out is None or out["ok"]) else 0], device=dev)
        dist.broadcast(flag, src=0)
        if out is None:
            out = {"ok": bool(flag.item())}
    del runner, op, dp, params
    torch.cuda.empty_cache()
    return out


def with_model_leg(args, wl, N, hp, lr_fn, world, rank, dev, dist):
    import torch
    from gaccum_b200.train_op import GaccumTrainOp
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bert_producer as bp
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    shape = {"bert_small": (8, 128), "bert_base": (32, 128), "bert_large": (4, 512)}[wl]
    torch.manual_seed(7)
    model = bp.Bert(wl).to(dev)
    named = bp.tf_names(model)
    params, names = [p for _, p in named], [n for n, _ in named]
    if world > 1 and args.dp == "fused":
        from gaccum_b200.distributed import FusedDataParallelTrainOp
        runner = FusedDataParallelTrainOp(params, names, hp, N, lr_fn, global_step=1)
    elif world > 1:
        from gaccum_b200.distributed import DataParallelTrainOp
        runner = DataParallelTrainOp(GaccumTrainOp(params, names, hp, N, lr_fn, global_step=1), None)
    else:
        runner = GaccumTrainOp(params, names, hp, N, lr_fn, global_step=1)
    gen = torch.Generator(device=dev); gen.manual_seed(100 + rank)
    batches = [bp.synthetic_batch(shape[0], shape[1], dev, gen) for _ in range(8)]
    stream = torch.cuda.current_stream(dev)
    t_op = [0.0]

    def step(i, timed=False):
        loss = model(*batches[i % 8]) / world                      # 04:46 loss / num_workers
        grads = torch.autograd.grad(loss, params)
        if timed:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream); runner.run(grads); b.record(stream)
            return a, b
        runner.run(grads)

    for i in range(2 * N):
        step(i)
    torch.cuda.synchronize(dev)
    if dist is not None:
        dist.barrier()
    Km = args.model_steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pairs = []
    e0.record(stream)
    for i in range(Km):
        pairs.append(step(i, timed=True))
    e1.record(stream)
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    op_ms = sum(a.elapsed_time(b) for a, b in pairs)
    if dist is not None:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return {"value": world * Km / (ms * 1e-3), "unit": "micro-steps/s", "steps": Km, "ms_per_step": ms / Km,
            "train_op_ms_per_step": op_ms / Km, "train_op_share": op_ms / ms,
            "producer": f"tools/bert_producer.py {wl} micro_bs={shape[0]} seq_len={shape[1]} fp32 params, TF32 matmuls, torch SDPA",
            "note": "forward/backward is plain PyTorch and is not part of this repository's path; it only supplies gradients"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="bert_small", choices=sorted(WORKLOADS))
    ap.add_argument("--accum-n", type=int, default=0)
    ap.add_argument("--sigma", type=float, default=1e-3, help="gradient std; 1e-3 clips at BERT-Small, 1e-4 does not")
    ap.add_argument("--dp", default="fused", choices=["fused", "allreduce"], help="multi-GPU exchange: in-kernel over peer memory, or NCCL all-reduce baseline")
    ap.add_argument("--no-launch-events", action="store_true", help="experiment: time only the whole region (no event between launches)")
    ap.add_argument("--no-clip", action="store_true", help="experiment: AdamWeightDecay without clip_by_global_norm (single-pass apply)")
    ap.add_argument("--model-steps", type=int, default=48, help="micro-steps of the with-model leg (0 disables)")
    ap.add_argument("--e2e-steps", type=int, default=48)
    ap.add_argument("--parity-steps", type=int, default=-1, help="micro-steps of the pre-timing parity self-check against the CPU oracle (-1: 2*min(N,4)+1, 0: skip)")
    ap.add_argument("--e2e-keep-affinity", action="store_true", help="experiment: keep the GPU-local CPU affinity for the whole e2e leg")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU-oracle timing (0 disables)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's parameters, optimizer state and stats as DIR/<name>.npy (--impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200: the reference arm times the CPU oracle, not the train_op")
    args.cpu_budget_given = any(a.startswith("--cpu-budget") for a in sys.argv[1:])
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
