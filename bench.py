#!/usr/bin/env python
"""bench.py -- env-steps/s of the b200sim CUDA path on the BASELINE.json workloads.

  python bench.py [--gpus N] [--steps K] [--warmup W]          our arm (one rank per GPU under torchrun for N > 1)
  python bench.py [...] --dump-outputs DIR                     ... and what its last timed step returned, as DIR/<name>.npy
  python bench.py --impl reference [...]                       the CPU arm: this repo's fp64 restatement of the
                                                               reference's mj_step path (the reference itself cannot
                                                               be imported: `mujoco`/`gymnasium` are absent), on all
                                                               host cores, on a bounded sample of the same workload

A "step" is one `step()` of every env of the batch (headline: FetchPickAndPlace-v4, 4096 envs per GPU, 20 physics sub-steps per
env-step, TimeLimit 50 with same-step autoreset so every counted env-step contains a physics step).  Rank 0 prints ONE JSON line:
the headline workload is `value` / `e2e` / `roofline`; the other BASELINE configs (3: Shadow Hand + 92 touch sensors, 4: AntMaze_Large
at 1024 envs per GPU, 5a: AdroitHandHammer, 5b: FrankaKitchen, and with >= 2 ranks 5: the Hammer + Kitchen mixed batch) are timed
AFTER the headline, outside its events, and reported in the `configs` array.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# stdout carries exactly ONE JSON line: NCCL's own banner ("NCCL version ...", printed on stdout when NCCL_DEBUG is set) goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
# ... and whatever else a library writes to file descriptor 1 ends up on stderr too: the JSON line is written to a duplicate of the
# original stdout
_JSON_FD = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_JSON_FD, (json.dumps(line) + "\n").encode())

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TASK, ENV_ID, ENVS_PER_GPU = "FetchPickAndPlace", "FetchPickAndPlace-v4", 4096
# algorithmic HBM bytes per env-step (SURVEY.md 8d): state read+write, action, obs/goals/reward/flags written
B_ALG = 2 * 4 * (22 + 2 * 21 + 2 + 7 + 3 + 1) + 4 * 4 + 4 * (25 + 2 * 3) + 10
# workloads (BASELINE.json configs): name -> (env id, action dim, sub-steps, algorithmic bytes per env-step, default envs/GPU)
WORKLOADS = {
    "fetch_pick_and_place": ("FetchPickAndPlace-v4", 4, 20, B_ALG, 4096),
    # config 3 (plain 61-dim observation; nq = 31, nv = 30 without the visual-only target body)
    "hand_block": ("HandManipulateBlockRotateXYZ-v1", 20, 20, 2 * 4 * (31 + 60 + 20 + 0 + 7 + 1) + 80 + 4 * (61 + 14) + 10, 2048),
    # config 3 as named: 24 DoF + 92 touch sensors (153-dim observation)
    "hand_block_touch": ("HandManipulateBlockRotateXYZ_ContinuousTouchSensors-v1", 20, 20,
                         2 * 4 * (31 + 60 + 20 + 0 + 7 + 1) + 80 + 4 * (153 + 14) + 10, 2048),
    # further env families on the same kernels (general convex collider: cylinder puck, ellipsoid egg)
    "fetch_slide": ("FetchSlide-v4", 4, 20, 2 * 4 * (22 + 2 * 21 + 0 + 7 + 3 + 1) + 4 * 4 + 4 * (25 + 2 * 3) + 10, 4096),
    "hand_egg": ("HandManipulateEggRotate-v1", 20, 20, 2 * 4 * (31 + 60 + 20 + 0 + 7 + 1) + 80 + 4 * (61 + 14) + 10, 2048),
    # config 5a: AdroitHandHammer (33 dofs, wide kernel build); registered id is -v2 (SURVEY.md 8, config-name caveats)
    "adroit_hammer": ("AdroitHandHammer-v2", 26, 5, 2 * 4 * (33 + 66 + 26 + 7 + 3 + 1) + 104 + 4 * (46 + 6) + 10, 2048),
    "adroit_relocate": ("AdroitHandRelocate-v2", 30, 5, 2 * 4 * (36 + 72 + 30 + 7 + 3 + 1) + 120 + 4 * (39 + 6) + 10, 2048),
    "adroit_pen": ("AdroitHandPen-v2", 24, 5, 2 * 4 * (30 + 60 + 24 + 7 + 3 + 1) + 96 + 4 * (45 + 6) + 10, 2048),
    "adroit_door": ("AdroitHandDoor-v2", 28, 5, 2 * 4 * (30 + 60 + 28 + 7 + 3 + 1) + 112 + 4 * (39 + 6) + 10, 2048),
    # config 5b: FrankaKitchen-v1 (csrc/b200sim_kitchen_groups.cu); 40 sub-steps per env-step
    "franka_kitchen": ("FrankaKitchen-v1", 9, 40, 2 * 4 * (30 + 2 * 29 + 9) + 36 + 4 * (59 + 2 * 30 + 2) + 4, 2048),
    "antmaze_large": ("AntMaze_Large-v5", 8, 5, 2 * 4 * (15 + 28 + 0 + 0 + 2 + 1) + 32 + 4 * (105 + 2 + 2) + 10, 1024),  # config 4: 8192 envs over 8 GPUs
}
# the BASELINE.json configs next to the headline (config 2), in the `configs` array of the default run
EXTRA_CONFIGS = [("3: Hand + 92 touch sensors", "hand_block_touch"), ("4: AntMaze_Large, 1024 envs/GPU (8192 over 8 GPUs)", "antmaze_large"),
                 ("5a: AdroitHandHammer", "adroit_hammer"), ("5b: FrankaKitchen", "franka_kitchen")]
FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # non-tensor FP32: 148 SMs x 128 lanes x 2 (FMA) x 1.965 GHz = 74.4


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------------------------------------------
# CPU arm: the fp64 oracle on all host cores -- persistent worker processes, K env-steps per message
def _cpu_worker(conn, nenv, seed0, native):
    import numpy as np

    from gymnasium_robotics_b200.models import load_model
    from oracle import oracle_sim
    from oracle.fetch_env import OracleFetchEnv

    if native:
        oracle_sim.use_native_build()
    model = load_model("fetch_pick_and_place")
    envs = [OracleFetchEnv(TASK, model=model) for _ in range(nenv)]
    for i, e in enumerate(envs):
        e.reset(seed=seed0 + i)
    t = [0] * nenv
    rng = np.random.default_rng(seed0)
    tape = rng.uniform(-1, 1, (64, nenv, 4))
    k = 0
    conn.send("ready")
    while True:
        nsteps = conn.recv()
        if nsteps <= 0:
            break
        for _ in range(nsteps):
            a = tape[k % 64]
            k += 1
            for i, e in enumerate(envs):
                e.step(a[i])
                t[i] += 1
                if t[i] >= 50:  # TimeLimit + autoreset, as in the GPU arm
                    e.reset()
                    t[i] = 0
        conn.send(nenv * nsteps)


def run_reference(args, quiet=False):
    import multiprocessing as mp

    from oracle import oracle_sim

    native = not args.portable_oracle
    if native:
        oracle_sim.use_native_build()   # gcc -O3 -march=native for THIS box, loaded in the parent too (visible to the driver)
    oracle_sim.lib()
    cores = max(1, os.cpu_count() or 1)
    per = max(1, max(args.sample_envs, 2 * cores) // cores)
    nenv = per * cores
    ctx = mp.get_context("fork")
    workers = []
    for w in range(cores):
        a, b = ctx.Pipe()
        p = ctx.Process(target=_cpu_worker, args=(b, per, 1000 * w, native), daemon=True)
        p.start()
        workers.append((p, a))
    for _, c in workers:
        assert c.recv() == "ready"

    def chunk(nsteps):
        t0 = time.perf_counter()
        for _, c in workers:
            c.send(nsteps)
        done = sum(c.recv() for _, c in workers)
        return done, time.perf_counter() - t0

    chunk(max(1, min(args.warmup, 3)))
    reps = min(max(3, args.reps), args.steps)
    rates = []
    for r in range(reps):   # args.steps env-steps in all, split as evenly as possible over the repetitions
        done, dt = chunk(args.steps // reps + (r < args.steps % reps))
        rates.append(done / dt)
    for p, c in workers:
        c.send(0)
    for p, c in workers:
        p.join(timeout=10)
    value = statistics.median(rates)
    sample = (f"{nenv} envs ({per} per worker process, {cores} processes) x {args.steps} env-steps over {reps} repetitions, "
              f"one IPC message per repetition, TimeLimit 50 + reset; liboracle built with {'-O3 -march=native' if native else '-O2'}")
    line = {"impl": "reference", "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * nenv / value,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{ENV_ID}, CPU restatement of the reference mj_step path (NOT MuJoCo: dependency absent), "
                                   f"bounded sample of {nenv} envs per step", "n_substeps": 20},
            "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample,
                             "median": value, "min": min(rates), "max": max(rates), "per_core": value / cores, "repetitions": reps},
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if not quiet:
        emit(line)
    return line


# ----------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


class Harness:
    """Process-wide pieces of the GPU arm: rank / device, the L2 flush buffer, the barrier."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback on the product path)")
        self.dev = torch.device(f"cuda:{self.local}")
        torch.cuda.set_device(self.dev)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        self.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=self.dev)  # > L2 (126 MB)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    def sum_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(x) for x in t.tolist()]


def make_env(H, workload, n, rng_mode):
    from gymnasium_robotics_b200.fetch import FetchVectorEnv

    env_id = WORKLOADS[workload][0]
    if workload == "fetch_pick_and_place":
        # --rng-mode device: resets drawn inside the library (b200sim_reset) with seeds invariant to the world size
        kw = dict(env_offset=H.rank * n) if rng_mode == "device" else {}
        env = FetchVectorEnv(TASK, num_envs=n, device=H.dev, rng_mode=rng_mode, autoreset_mode="same_step", **kw)
    else:
        import gymnasium_robotics_b200 as grb

        env = grb.make_vec(env_id, num_envs=n, device=H.dev, rng_mode="torch", autoreset_mode="same_step")
    env.reset(seed=0 if rng_mode == "device" else 1000 * H.rank)  # seeds seed0 + global env index would need numpy streams; device RNG is per rank
    return env


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def step_outputs(result):
    """What env.step returned -- observation entries, reward, terminated, truncated and the tensors of the info dict (nested keys
    joined with '.', info keys prefixed 'info.') -- as host arrays: float64 stays float64, integers become float64 (exact for the
    int32 solver counters), everything else float32."""
    import numpy as np
    import torch

    obs, reward, terminated, truncated, info = result
    out = {}

    def add(name, v):
        if isinstance(v, dict):
            for k, x in v.items():
                add(f"{name}.{k}" if name else k, x)
        elif torch.is_tensor(v):
            a = v.detach().cpu().numpy()
            out[name] = a.astype(np.float64 if a.dtype == np.float64 or a.dtype.kind in "iu" else np.float32)

    add("" if isinstance(obs, dict) else "obs", obs)
    add("reward", reward)
    add("terminated", terminated)
    add("truncated", truncated)
    add("info", info)
    return out


def write_outputs(arrays, n, path):
    """DIR/<name>.npy for every array; above DUMP_LIMIT_BYTES in all, the rows of a fixed seeded sample of the n envs (their indices
    in env_index.npy) of every array whose first axis is the env axis."""
    import numpy as np

    budget = DUMP_LIMIT_BYTES - 1024 * (len(arrays) + 1)   # a .npy header takes at most 1 KB
    total = sum(a.nbytes for a in arrays.values())
    if total > budget:
        per_env = sum(a.nbytes for a in arrays.values() if a.ndim and a.shape[0] == n) / n
        fixed = total - per_env * n
        keep = int((budget - fixed) // (per_env + 8))   # + 8 bytes per kept env: its float64 index
        if keep < 1:
            raise SystemExit(f"--dump-outputs: the outputs do not fit in {DUMP_LIMIT_BYTES} bytes")
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: a[idx] if a.ndim and a.shape[0] == n else a for k, a in arrays.items()}
        arrays["env_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def time_workload(H, workload, n, steps, warmup, rng_mode="torch", nvtx=False, sample_clocks=False, gather=False, keep_outputs=False):
    """Three timed arms over the same env: (1) `value`: CUDA events around env.step with device-resident actions, (2) the step
    kernel alone, (3) end to end with HOST buffers -- pinned actions H2D, the packed result rows D2H, every step.  All times are
    per-rank sums; the caller takes the max over ranks.  keep_outputs: res["outputs"] holds what the last step of arm (1) returned
    (step_outputs)."""
    torch = H.torch
    env_id, nact, nsub, b_alg, _ = WORKLOADS[workload]
    env = make_env(H, workload, n, rng_mode)
    g = torch.Generator(device=H.dev).manual_seed(1234 + H.rank)
    tape = torch.rand((64, n, nact), generator=g, device=H.dev) * 2 - 1  # pre-generated action tape (RNG outside the timed region)
    flush = H.flush
    # ---- device-resident arm
    for k in range(warmup):
        env.step(tape[k % 64])
    H.barrier()
    sampler = ClockSampler(H.local) if (sample_clocks and H.rank == 0) else None
    if sampler:
        sampler.start()
    launches0 = env.backend.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    nv = torch.cuda.nvtx if nvtx else None   # --nvtx: ranges for ncu --nvtx filtering (SURVEY.md section 5, tracing)
    reset_masks = []
    for k in range(steps):
        flush.fill_(float(k))  # evict L2 between timed iterations (outside the timed interval)
        ev[k][0].record()
        if nv:
            nv.range_push(f"env.step {k}")
        last = env.step(tape[k % 64])
        if nv:
            nv.range_pop()
        ev[k][1].record()
        info = last[4]
        if "_final_obs" in info:
            reset_masks.append(info["_final_obs"])   # same-step autoreset happened inside this timed step
    H.barrier()
    outputs = step_outputs(last) if keep_outputs else None   # before the arms below step the env again
    ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = env.backend.launches - launches0
    resets = int(sum(int(m.sum()) for m in reset_masks))
    # ---- dominant kernel alone (the step kernel), same stream, CUDA events around the launch only
    out = env.backend.new_outputs()
    kitchen = workload == "franka_kitchen"
    for k in range(steps):
        # kitchen: the kernel's input is a position target; it is derived exactly as env.step derives it (velocity-limited step from
        # the last robot pose, kitchen.py control_targets) OUTSIDE the timed events, so the kernel arm sees the contact load of the
        # `value` arm instead of an arm resting at its initial pose
        kact = env.control_targets(tape[k % 64]) if kitchen else tape[k % 64]
        flush.fill_(float(k))
        kev[k][0].record()
        env.backend.step(kact, out)
        kev[k][1].record()
        if kitchen:
            env._last_robot_qpos = out["obs"][:, :9].clone()
    H.barrier()
    kms = sum(a.elapsed_time(b) for a, b in kev) / steps
    clocks = sampler.stop() if sampler else None
    # ---- end to end through the public API with HOST buffers: pinned actions H2D, ONE packed row per env D2H, every step
    env.reset(seed=1000 * H.rank + 7)
    host_tape = [tape[k].cpu().pin_memory() for k in range(8)]
    packed_mode = workload != "franka_kitchen"   # the kitchen's observation gets its noise after the kernel: copied as separate tensors
    if packed_mode:
        host_out = [torch.empty((n, env.backend.packed_w), dtype=torch.float32).pin_memory()]
    else:
        host_out = [torch.empty((n, env.task.nobs), dtype=torch.float32).pin_memory(), torch.empty(n, dtype=torch.float32).pin_memory(),
                    torch.empty(n, dtype=torch.bool).pin_memory(), torch.empty(n, dtype=torch.bool).pin_memory()]
    h2d = n * nact * 4
    d2h = sum(v.numel() * v.element_size() for v in host_out)
    gatherer = None
    if gather and H.world > 1 and packed_mode:
        from gymnasium_robotics_b200.sharding import PackedGather

        gatherer = PackedGather(n, env.backend.packed_w, H.dev)

    def e2e_step(k, with_gather):
        o, r, te, tr, info = env.step(host_tape[k % 8])  # the vector env copies the pinned host actions to the device
        if packed_mode:
            p = env._last["packed"]
            host_out[0].copy_(p, non_blocking=True)
            if with_gather:
                gatherer.launch(p)     # NCCL all-gather of the packed rows on a side stream: overlaps the next step's kernel
        else:
            host_out[0].copy_(o["observation"], non_blocking=True)
            host_out[1].copy_(r, non_blocking=True)
            host_out[2].copy_(te, non_blocking=True)
            host_out[3].copy_(tr, non_blocking=True)
        torch.cuda.current_stream(H.dev).synchronize()

    def e2e_arm(with_gather):
        for k in range(warmup):
            e2e_step(k, with_gather)
        if with_gather:
            gatherer.wait()
        H.barrier()
        tot = 0.0
        for k in range(steps):
            flush.fill_(float(k))
            torch.cuda.synchronize(H.dev)
            t0 = time.perf_counter()
            e2e_step(k, with_gather)
            tot += time.perf_counter() - t0
        if with_gather:
            t0 = time.perf_counter()
            gatherer.wait()               # the last gather has nothing to hide behind: counted
            tot += time.perf_counter() - t0
        H.barrier()
        return tot

    e2e_s = e2e_arm(False)
    e2e_gather_s = e2e_arm(True) if gatherer is not None else None
    res = dict(workload=workload, env_id=env_id, n=n, nsub=nsub, nact=nact, b_alg=b_alg, ms=ms, kms=kms, e2e_ms=e2e_s * 1e3,
               e2e_gather_ms=None if e2e_gather_s is None else e2e_gather_s * 1e3, launches=launches, resets=resets, h2d=h2d, d2h=d2h,
               clocks=clocks, overflow_env_steps=int(env.backend.overflow_counter[0]),
               wpb=None, gathered_rows=None if gatherer is None else int(gatherer.rows), outputs=outputs)
    env.close()
    return res


def roofline_object(res, steps):
    peak, how = measured_peaks()
    kms, n, b_alg = res["kms"], res["n"], res["b_alg"]
    achieved = b_alg * n / (kms / 1e3) / 1e9
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
            "peak_source": how, "algorithmic_bytes_per_env_step": b_alg, "kernel_ms": kms,
            "note": "path is FP32-issue/latency bound (SURVEY.md 0.4, 8d); HBM fraction is reported because the metric asks for it; "
                    "the compute-side figures below come from the committed ncu capture named in `ncu_source`"}
    # compute-side figures (BASELINE.md section 4, SURVEY.md 8d) from the committed ncu summary of this workload's kernel
    p = os.path.join(ROOT, "profiles", f"roofline_{res['workload']}.json")
    if os.path.exists(p):
        d = json.load(open(p))
        roof["traffic"] = d.get("dram_bytes_per_launch")
        for k in ("issue_active_pct", "warps_active_pct", "fma_pipe_pct", "avg_active_lanes", "top_stalls", "local_load_store_inst",
                  "registers_per_thread", "smem_per_block_bytes", "ncu_source", "ncu_kernel_ms"):
            if k in d:
                roof[k] = d[k]
        if d.get("fp32_flop_per_launch"):
            # executed FP32 flops of the captured launch (fadd + fmul + 2 ffma, ncu) at THIS run's kernel time
            roof["fp32_flop_per_env_step"] = d["fp32_flop_per_launch"] / d.get("envs_per_launch", n)
            roof["fp32_tflops"] = d["fp32_flop_per_launch"] * (n / d.get("envs_per_launch", n)) / (kms / 1e3) / 1e12
            roof["fp32_peak_tflops"] = FP32_PEAK_TFLOPS
            roof["fp32_frac"] = roof["fp32_tflops"] / FP32_PEAK_TFLOPS
    return roof


def run_ours(args):
    H = Harness()
    world, rank = H.world, H.rank
    mixed = None
    headline = args.workload
    if args.workload == "mixed_hammer_kitchen":
        # BASELINE config 5: heterogeneous batch, whole ranks per model (sharding.mixed_batch_assignment), 1 024 envs per GPU; the
        # line reports the aggregate over both models, the roofline object is rank 0's model (the Hammer)
        from gymnasium_robotics_b200.sharding import mixed_batch_assignment

        if world < 2:
            raise SystemExit("--workload mixed_hammer_kitchen needs at least 2 ranks (torchrun --nproc-per-node 2|4|8)")
        mixed = mixed_batch_assignment(["adroit_hammer", "franka_kitchen"], world)
        headline = mixed[rank]
        args.envs_per_gpu = args.envs_per_gpu or 1024
    n = args.envs_per_gpu or WORKLOADS[headline][4]
    res = time_workload(H, headline, n, args.steps, args.warmup, rng_mode=args.rng_mode, nvtx=args.nvtx, sample_clocks=True, gather=args.gather,
                        keep_outputs=bool(args.dump_outputs) and rank == 0)
    if os.environ.get("B200SIM_BENCH_DEBUG"):
        print(f"[rank {rank}] ms/step {res['ms'] / args.steps:.3f} kernel {res['kms']:.3f} e2e {res['e2e_ms'] / args.steps:.3f}", file=sys.stderr)
    ms, e2e_ms, kms, e2e_g = H.max_over_ranks([res["ms"], res["e2e_ms"], res["kms"], res["e2e_gather_ms"] or 0.0])
    resets, overflow = H.sum_over_ranks([res["resets"], res["overflow_env_steps"]])
    total_envs = n * world
    value = total_envs * args.steps / (ms / 1e3)
    e2e_value = total_envs * args.steps / (e2e_ms / 1e3)
    # ---- the other BASELINE configs, after the headline and outside its timed region (default run only)
    configs = []
    if args.workload == "fetch_pick_and_place" and not args.no_configs and args.envs_per_gpu is None:
        ksteps, kwarm = min(args.steps, args.config_steps), 3
        plan = list(EXTRA_CONFIGS)
        for label, wl in plan:
            cn = WORKLOADS[wl][4]
            r = time_workload(H, wl, cn, ksteps, kwarm)
            cms, ce2e, ckms = H.max_over_ranks([r["ms"], r["e2e_ms"], r["kms"]])
            cres, = H.sum_over_ranks([r["resets"]])
            configs.append({"config": label, "workload": f"{r['env_id']}, {cn} envs/GPU x {world} GPU(s), {r['nsub']} sub-steps/env-step",
                            "value": cn * world * ksteps / (cms / 1e3), "unit": "env-steps/s", "steps": ksteps, "warmup": kwarm,
                            "ms_per_step": cms / ksteps, "kernel_ms": ckms,
                            "e2e": {"value": cn * world * ksteps / (ce2e / 1e3), "unit": "env-steps/s", "h2d_bytes_per_step": r["h2d"],
                                    "d2h_bytes_per_step": r["d2h"]},
                            "gpu_launches": r["launches"], "resets_in_timed_region": int(cres),
                            "roofline": {k: v for k, v in roofline_object(r, ksteps).items() if k != "note"}})
        if world >= 2:
            from gymnasium_robotics_b200.sharding import mixed_batch_assignment

            assign = mixed_batch_assignment(["adroit_hammer", "franka_kitchen"], world)
            r = time_workload(H, assign[rank], 1024, ksteps, kwarm)
            cms, ce2e = H.max_over_ranks([r["ms"], r["e2e_ms"]])
            configs.append({"config": "5: AdroitHandHammer + FrankaKitchen mixed batch, whole ranks per model",
                            "workload": f"1024 envs/GPU x {world} GPUs, models per rank: {assign}", "value": 1024 * world * ksteps / (cms / 1e3),
                            "unit": "env-steps/s", "steps": ksteps, "warmup": kwarm, "ms_per_step": cms / ksteps,
                            "e2e": {"value": 1024 * world * ksteps / (ce2e / 1e3), "unit": "env-steps/s", "h2d_bytes_per_step": r["h2d"],
                                    "d2h_bytes_per_step": r["d2h"]}})
    if rank == 0:
        if args.dump_outputs:
            write_outputs(res["outputs"], n, args.dump_outputs)
        env_id, nsub = res["env_id"], res["nsub"]
        cpu = None
        if world == 1 and not args.no_cpu_baseline and args.workload == "fetch_pick_and_place":
            cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "24", "--warmup", "2"]
            try:
                outp = subprocess.run(cmd, capture_output=True, text=True, timeout=600).stdout.strip().splitlines()
                cpu = json.loads(outp[-1])["cpu_baseline"]
            except Exception as e:  # noqa: BLE001
                cpu = {"value": None, "unit": "env-steps/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
        e2e = {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": res["h2d"], "d2h_bytes_per_step": res["d2h"],
               "ms_per_step": e2e_ms / args.steps, "d2h_copies_per_step": 1 if args.workload != "franka_kitchen" else 4}
        if res["e2e_gather_ms"] is not None:
            e2e["with_gather"] = {"value": total_envs * args.steps / (e2e_g / 1e3), "ms_per_step": e2e_g / args.steps,
                                  "collective": "NCCL all_gather_into_tensor of the packed rows on a side stream (sharding.PackedGather)",
                                  "rows_on_every_rank": res["gathered_rows"], "bytes_per_rank_per_step": res["d2h"]}
        line = {"metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": ("AdroitHandHammer-v2 + FrankaKitchen-v1 mixed batch, whole ranks per model; rank 0: " if mixed else "") +
                                       f"{env_id}, {n} envs/GPU, {nsub} sub-steps/env-step, random actions U(-1,1), TimeLimit, "
                                       "same-step autoreset", "envs_per_gpu": n, "l2": "flushed between timed iterations (256 MB fill)",
                           "parallelism": f"env-sharded x{world}, no data-path collective" + (f"; models per rank: {mixed}" if mixed else ""),
                           "reset_rng": "in-kernel Philox (b200sim_reset)" if args.rng_mode == "device" else "torch device generator"},
                "roofline": roofline_object(res, args.steps), "cpu_baseline": cpu, "e2e": e2e,
                "gpu_launches": res["launches"], "resets_in_timed_region": int(resets), "solver_overflow_env_steps": int(overflow),
                "clocks": res["clocks"], "configs": configs}
        emit(line)
    if world > 1:
        H.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=None)
    ap.add_argument("--workload", default="fetch_pick_and_place", choices=sorted(WORKLOADS) + ["mixed_hammer_kitchen"])
    ap.add_argument("--sample-envs", type=int, default=256, help="envs per step of the CPU arm's bounded sample")
    ap.add_argument("--reps", type=int, default=3, help="repetitions of the CPU arm (median reported)")
    ap.add_argument("--portable-oracle", action="store_true", help="CPU arm: use the -O2 oracle build instead of -O3 -march=native")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` array (the other BASELINE configs)")
    ap.add_argument("--config-steps", type=int, default=20, help="timed steps of each entry of the `configs` array")
    ap.add_argument("--gather", action="store_true", help="N > 1: also time e2e with the NCCL all-gather of the packed rows")
    ap.add_argument("--nvtx", action="store_true", help="NVTX range around every timed env.step (profiling runs only)")
    ap.add_argument("--rng-mode", default="torch", choices=["torch", "device"],
                    help="reset draws of the Fetch workload: torch's device generator (default) or in-kernel (b200sim_reset)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline workload returned as DIR/<name>.npy (rank 0's envs; "
                         "at most 64 MB, a fixed sample of the envs above that); the inputs are seeded, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        if int(os.environ.get("RANK", "0")) == 0:
            run_reference(args)
        return
    run_ours(args)


if __name__ == "__main__":
    main()
