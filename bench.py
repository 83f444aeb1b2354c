#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native BlueSky-Gym step path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload at every N (weak scaling): BASELINE.json configs[1] per GPU -- HorizontalCREnv-v0, 4096 env
instances, 20 intruders each (21 aircraft), StateBased conflict detection in every simulator substep,
10 substeps of DT 5 s per env step, autoreset, random actions resident in HBM.  One "step" = one
batched env step = one launch of the env-step megakernel over all envs of the rank.
Metric: env-steps/s, whole job.  Extra: CD aircraft-pairs/s at N = 100k (BASELINE configs[4]).

Prints ONE JSON line (rank 0).  `--impl reference` times the CPU restatement of the reference's step
loop (oracle/, "port": the reference's own BlueSky dependency is not installable here) on the host cores.
`--dump-outputs DIR` writes what the last timed step returned on rank 0 (obs keys, reward, terminated, truncated of
every env, float32) as DIR/<name>.npy: the inputs depend only on the arguments, so two builds can be compared.
"""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
N_INTRUDERS = 20
N_SUB = 10
CD_N = 100_000
PREROLL_STEPS = 150        # untimed env steps before the warm-up: episodes desynchronised (stationary regime)
# algorithmic work (SURVEY.md section 8d; restated in DESIGN.md)
F_PAIR = 67.0            # FP32 flop per ordered aircraft pair of state-based CD
F_KIN = 250.0            # FP32 flop per aircraft-substep of Traffic.update
F_OBS = 3000.0           # per env step
A = N_INTRUDERS + 1
FLOP_PER_ENV_STEP = N_SUB * (A * F_KIN + A * (A - 1) * F_PAIR) + F_OBS
BYTES_PER_ENV_STEP = 2 * A * 68 + (5 * N_INTRUDERS + 3) * 4 + 2 * (4 * 8 + 4 * 4 + 16 * 4) + 6 * 4 + 10


# ------------------------------------------------------------------------------------------------ CPU arm
def _cpu_worker(args):
    """One host core stepping oracle envs (the restated reference step loop) for `budget` seconds."""
    seed, budget = args
    sys.path.insert(0, ROOT)
    from oracle import envs as oenvs
    np.random.seed(seed)
    env = oenvs.HorizontalCREnv(n_intruders=N_INTRUDERS, cd_enabled=True)
    env.reset()
    rng = np.random.default_rng(seed)
    for _ in range(3):
        env.step(rng.uniform(-1, 1, 1))
    n, t0, ep = 0, time.perf_counter(), 0
    while time.perf_counter() - t0 < budget:
        _, _, term, _, _ = env.step(rng.uniform(-1, 1, 1))
        n += 1
        ep += 1
        if term or ep >= 300:
            env.reset()
            ep = 0
    return n, time.perf_counter() - t0


_OUT = sys.stdout


def cpu_baseline(budget_s=12.0, cores=None):
    cores = cores or os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        res = pool.map(_cpu_worker, [(1000 + i, budget_s) for i in range(cores)])
    steps = sum(r[0] for r in res)
    wall = max(r[1] for r in res)
    return dict(value=steps / wall, unit="env-steps/s", cores=cores, kind="port",
                sample=f"{steps} env steps of HorizontalCREnv-v0 (20 intruders, CD on) in {wall:.1f} s, "
                       f"one oracle env per process, {cores} processes")


def _real_reference_env(seed):
    """The UNMODIFIED reference env (real bluesky-simulator + gymnasium from baseline/_ref) in the bench's configuration:
    20 intruders (module constant, horizontal_cr_env.py:17) and ASAS switched on."""
    sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
    import bluesky as bs
    import gymnasium as gym
    import bluesky_gym
    import bluesky_gym.envs.horizontal_cr_env as ref_env
    ref_env.NUM_INTRUDERS = N_INTRUDERS
    bluesky_gym.register_envs()
    env = gym.make("HorizontalCREnv-v0", render_mode=None)

    class Shim:
        def reset(self):
            out = env.reset(seed=seed)
            bs.stack.stack("ASAS ON")
            return out

        def step(self, a):
            o, r, term, trunc, i = env.step(a)
            return o, r, term or trunc, False, i
    return Shim()


def _ref_arm_worker(args):
    """One host core of the reference arm: `n_warm` untimed + `n_timed` timed env steps of one env (the oracle port, or the
    real reference stack when `real`)."""
    seed, n_warm, n_timed, real = args
    sys.path.insert(0, ROOT)
    if real:
        env = _real_reference_env(seed)
    else:
        from oracle import envs as oenvs
        np.random.seed(seed)
        env = oenvs.HorizontalCREnv(n_intruders=N_INTRUDERS, cd_enabled=True)
    env.reset()
    rng = np.random.default_rng(seed)
    ep, t0 = 0, 0.0
    for k in range(n_warm + n_timed):
        if k == n_warm:
            t0 = time.perf_counter()
        _, _, term, _, _ = env.step(rng.uniform(-1, 1, 1))
        ep += 1
        if term or ep >= 300:
            env.reset()
            ep = 0
    return n_timed, time.perf_counter() - t0


def probe_real_reference():
    """Is the reference's own stack importable from baseline/_ref (driver-provided on some pods)?  Returns None or a
    one-line reason why not."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(ref):
        return "baseline/_ref absent"
    code = ("import sys; sys.path.insert(0, %r); import bluesky, gymnasium, bluesky_gym, bluesky_gym.envs.horizontal_cr_env" % ref)
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    return None if p.returncode == 0 else (p.stderr.strip().splitlines() or ["import failed"])[-1][:200]


def run_reference(args):
    """Reference arm of the bench contract: the reference's CPU step loop on every host core.  One "step" of this arm = every
    core advances its own env by `per_step` env steps; W warm-up steps, then exactly K timed ones; value = env steps of all
    cores / the slowest core's wall time."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    why_not = probe_real_reference()
    real = why_not is None
    K, W = args.steps, max(0, args.warmup)
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        try:
            cal = pool.map(_ref_arm_worker, [(7, 1, 4, real)])[0]           # calibration: seconds per env step on one core
        except Exception as ex:
            real, why_not = False, repr(ex)[:200]
            cal = pool.map(_ref_arm_worker, [(7, 1, 4, False)])[0]
        t_step = cal[1] / cal[0]
        per_step = int(min(64, max(1, round(12.0 / (K * t_step)))))         # ~12 s of timed work per core
        res = pool.map(_ref_arm_worker, [(1000 + i, W * per_step, K * per_step, real) for i in range(cores)])
    steps, wall = sum(r[0] for r in res), max(r[1] for r in res)
    cb = dict(value=steps / wall, unit="env-steps/s", cores=cores, kind="reference" if real else "port",
              sample=f"{steps} env steps of HorizontalCREnv-v0 (20 intruders, CD on) in {wall:.1f} s: {cores} processes x {K} steps x "
                     f"{per_step} env steps, " + ("the reference's own env on real BlueSky (baseline/_ref)" if real else
                                                  "one oracle env per process"))
    if not real:
        cb["real_reference"] = f"not used: {why_not}"
    line = {"impl": "reference", "metric": "env_steps_per_sec", "value": cb["value"], "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": 1e3 * wall / K,
            "step_definition": f"every host core advances its env by {per_step} env steps ({cores * per_step} env steps per step)",
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.gpus), "cpu_baseline": cb, "gpu_launches": 0,
            "e2e": {"value": cb["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=_OUT, flush=True)


def workload_config(n_gpus):
    return {"workload": "HorizontalCREnv-v0 batched (BASELINE configs[1])", "envs_per_gpu": ENVS_PER_GPU,
            "envs_total": ENVS_PER_GPU * n_gpus, "n_intruders": N_INTRUDERS, "aircraft_per_env": A,
            "substeps_per_step": N_SUB, "simdt_s": 5.0, "cd": "StateBased every substep", "autoreset": "same_step",
            "max_episode_steps": 300, "preroll_steps": PREROLL_STEPS, "actions": "U(-1,1) float32, resident in HBM", "l2": "flushed between timed steps",
            "parallelism": f"env-sharded x{n_gpus}, no data-path collective"}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: NVML every ~2 ms (an nvidia-smi process
    per sample would be slower than the whole region), nvidia-smi only when NVML is unavailable."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index=0):
        self.samples, self.stop, self.index = [], False, index
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.bits = [pynvml.nvmlClocksEventReasonHwSlowdown, pynvml.nvmlClocksEventReasonHwThermalSlowdown,
                         pynvml.nvmlClocksEventReasonSwThermalSlowdown, pynvml.nvmlClocksEventReasonSwPowerCap]
            self.nvml = pynvml
        except Exception:
            self.nvml = None
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop:
            try:
                if self.nvml is not None:
                    mhz = float(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
                    r = int(self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                    self.samples.append([mhz, self.max_mhz] + [bool(r & b) for b in self.bits])
                    time.sleep(0.0005)
                    continue
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    f = [x.strip() for x in out.split(",")]
                    self.samples.append([float(f[0]), float(f[1])] + [x.lower().startswith("active") for x in f[2:6]])
            except Exception:
                pass
            time.sleep(0.05)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(s[0] for s in self.samples)
        reasons = [n for i, n in enumerate(self.NAMES) if any(s[2 + i] for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.samples[0][1], "reasons": reasons,
                "samples": len(self.samples), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def pin_to_gpu_numa_node(index):
    """One process per GPU: run this rank's host thread on the cores of the NUMA node its GPU hangs off, so the pinned
    blocks it allocates (first touch) and the Python loop that fills / reads them sit next to the PCIe root of the GPU.
    Returns a short description for the JSON line, or None when the topology cannot be read (then nothing is changed)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = int(vis.split(",")[index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else index
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:                      # NVML prints an 8-digit PCI domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        ids &= os.sched_getaffinity(0)
        if not ids:
            return None
        os.sched_setaffinity(0, ids)
        return f"numa node {node} ({len(ids)} cores)"
    except Exception:
        return None


# ------------------------------------------------------------------------------------------------ GPU arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    from bluesky_gym_sasha_b200 import _lib, build
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    from bluesky_gym_sasha_b200.vector_env import BlueSkyVectorEnv

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = pin_to_gpu_numa_node(local) if world > 1 else None     # each rank's host thread + pinned blocks next to its GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        build.build()
    if world > 1:
        dist.barrier()
    lib = _lib.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    E, K, W = ENVS_PER_GPU, args.steps, max(3, args.warmup)
    venv = BlueSkyVectorEnv("HorizontalCREnv-v0", E, device=local, seed=0, cd_enabled=True, n_intruders=N_INTRUDERS,
                            autoreset_mode="same_step", env_id_offset=rank * E)
    venv.reset_torch()
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    bank = torch.rand((K + W, E, 1), generator=g, device=dev) * 2.0 - 1.0      # actions resident in HBM
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MB > 126 MB L2
    # set-up: the env population is advanced to its stationary regime (episodes of different lengths: ~3 % of the envs finish
    # and re-generate their scenario in any step, ownships anywhere between the first turn and the waypoint) -- what a
    # training run sees after its first seconds; straight after reset() every env would be in the first steps of its first
    # episode at once.  Untimed, before the W warm-up steps; named in config.preroll_steps.
    for i in range(PREROLL_STEPS):
        venv.step_torch(bank[i % (K + W)])
    for i in range(W):
        venv.step_torch(bank[i])
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    launches0 = venv.gpu_launches
    with ClockSampler(local) as clk:
        # the device starts ~60 us per step behind the host, so that every timed interval is a kernel that was already
        # queued when its start event was reached: the figure is the device's, whatever the host's submission rate is
        # (8 ranks sharing one host submit slower than one)
        torch.cuda._sleep(int(min(K, 1000) * 60e-6 * 1.9e9))
        for i in range(K):
            flush.fill_(float(i))                           # evict the sim state from L2 (not timed)
            ev[i][0].record()
            out = venv.step_torch(bank[W + i])
            ev[i][1].record()
        barrier()
    launches = venv.gpu_launches - launches0
    dumped = step_outputs(*out) if args.dump_outputs and rank == 0 else None     # (the next step overwrites them)
    t_dev = sum(a.elapsed_time(b) for a, b in ev) * 1e-3
    t_dev = max_over_ranks(t_dev)
    value = E * world * K / t_dev
    kernel_ms = 1e3 * t_dev / K

    # back-to-back (L2-warm) figure, for context
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        venv.step_torch(bank[W + i])
    e1.record()
    barrier()
    warm_value = E * world * K / max_over_ranks(e0.elapsed_time(e1) * 1e-3)

    # end to end through the public numpy API: pinned host actions in, obs/reward/flags/info out, every step
    host_actions = bank[W:].cpu().numpy()
    for i in range(3):
        obs, rew, term, trunc, info = venv.step(host_actions[i % K])       # (results held like in the timed loop)
    barrier()
    prof = None
    if os.environ.get("BSG_BENCH_PROFILE"):      # where does the host time of the e2e loop go? (stats to stderr)
        import cProfile
        prof = cProfile.Profile()
        prof.enable()
    t0 = time.perf_counter()
    step_s = []
    for i in range(K):
        t1 = time.perf_counter()
        obs, rew, term, trunc, info = venv.step(host_actions[i])
        step_s.append(time.perf_counter() - t1)
    barrier()
    t_e2e = max_over_ranks(time.perf_counter() - t0)
    if prof is not None:
        import pstats
        prof.disable()
        pstats.Stats(prof, stream=sys.stderr).sort_stats("cumulative").print_stats(18)
    L = venv.layout
    h2d = E * L.act_dim * 4
    d2h = venv._out_bytes          # the mirrored head of the output block: obs, reward, info, flags, terminal-obs window
    ss = sorted(step_s)
    e2e = {"value": E * world * K / t_e2e, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "us_per_step_median": 1e6 * ss[len(ss) // 2], "us_per_step_max": 1e6 * ss[-1],
           "api": "BlueSkyVectorEnv.step, default arguments (numpy in; float32 numpy arrays out that the caller owns; "
                  "bsg_step_host_block: one H2D, one launch, one D2H of the output block straight into a pinned block leased to "
                  "the caller until the arrays are dropped -- no host copy)"}
    # same call with copy=False (views of two rotating pinned buffers instead of fresh copies), for context
    venv.copy = False
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        venv.step(host_actions[i])
    barrier()
    e2e["host_affinity"] = affinity
    e2e["value_copy_false"] = E * world * K / max_over_ranks(time.perf_counter() - t0)
    venv.copy = True
    # same call returning float64 observations (the dtype the reference's spaces declare; what the scalar gym.make envs return)
    venv.obs_dtype = np.dtype(np.float64)
    for i in range(3):
        venv.step(host_actions[i % K])
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        venv.step(host_actions[i])
    barrier()
    e2e["value_f64"] = E * world * K / max_over_ranks(time.perf_counter() - t0)
    venv.obs_dtype = np.dtype(np.float32)

    # single airspace, rows sharded over the ranks after one NCCL all-gather (BASELINE configs[4])
    cd_sharded = bench_cd_sharded(torch, dist, dev, StateBasedCD, world, rank, max_over_ranks, barrier) if world > 1 else None
    # one airspace with routes + MVP, its aircraft sharded over the ranks (SURVEY 8e + 8f-4)
    traffic_sharded = bench_traffic_sharded(torch, dist, dev, world, rank, max_over_ranks, barrier) if world > 1 else None

    # the other BASELINE configs: every rank steps its shard (env-sharded like the headline; max over ranks)
    legs = {name: bench_env_leg(torch, dev, BlueSkyVectorEnv, env_id, E_, kw, world, rank, max_over_ranks, barrier)
            for name, env_id, E_, kw in CONFIG_LEGS}
    other = None
    if world == 1:
        other = {name: bench_env_leg(torch, dev, BlueSkyVectorEnv, env_id, E_, kw, 1, 0, max_over_ranks, barrier)
                 for name, env_id, E_, kw in CONTEXT_LEGS}

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    line = None
    if rank == 0:
        fp32 = C_double_probe(lib, local)
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        achieved_tf = FLOP_PER_ENV_STEP * E / (kernel_ms * 1e-3) / 1e12
        traffic, traffic_src = None, None
        try:        # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed --set full capture
            tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["env_kernel<1, 32, 0>"]
            traffic, traffic_src = tr["dram_bytes_read"] + tr["dram_bytes_write"], "profiles/ncu_traffic.json <- " + tr["source"]
        except Exception:
            pass
        roof = {"bound": "fp32", "achieved": achieved_tf, "peak": fp32 / 1e12, "unit": "TFLOP/s",
                "frac": achieved_tf / (fp32 / 1e12), "traffic": traffic, "traffic_unit": "bytes per launch (DRAM)",
                "traffic_source": traffic_src, "kernel": "env_kernel<HorizontalCR,32,no wind>",
                "peak_source": "bsg_probe_fp32 (dense FFMA, measured in this run)",
                "flop_per_env_step": FLOP_PER_ENV_STEP,
                "note": "achieved = algorithmic flops (every ordered pair, every substep) / time; the in-group CD evaluates "
                        "exactly only the pairs its conservative filters keep (dcpa < R, not past the zone, entry within the "
                        "look-ahead) and keeps the intruder-intruder candidate list across the substeps of an env step "
                        "while velocities hold: results bit-identical to cd_enabled=2 (filter redone every substep)",
                "hbm": {"achieved": BYTES_PER_ENV_STEP * E / (kernel_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback",
                        "bytes_per_env_step": BYTES_PER_ENV_STEP}}
        # CD at N = 100k on this GPU (BASELINE configs[4], single-GPU share)
        cd = bench_cd(torch, dev, StateBasedCD, fp32)
        traffic_leg = bench_traffic(torch, dev, hbm_peak) if world == 1 else None
        cb = None if (args.skip_cpu or world > 1) else cpu_baseline(budget_s=10.0)
        # compact headline of the second BASELINE metric, early in the line (the full records follow at the end)
        cd_head = {"n_aircraft": cd["n_aircraft"], "ordered_pairs_per_s": cd["ordered_pairs_per_s"], "ms": cd["ms"],
                   "frac_of_fp32_peak": cd["roofline"]["frac"], "form": "every ordered pair, 1 GPU"}
        if cd_sharded is not None:
            cd_sharded["roofline_frac_per_gpu"] = cd_sharded["ordered_pairs_per_s"] * F_PAIR / world / fp32
            cd_head.update({"sharded_ordered_pairs_per_s": cd_sharded["ordered_pairs_per_s"], "sharded_ms": cd_sharded["ms"],
                            "sharded_frac_of_fp32_peak_per_gpu": cd_sharded["roofline_frac_per_gpu"],
                            "sharded_form": f"rows over {world} GPUs after one NCCL all-gather, every ordered pair"})
            if "symmetric_dealt" in cd_sharded:
                cd_head.update({"sharded_symmetric_ordered_pairs_per_s": cd_sharded["symmetric_dealt"]["ordered_pairs_per_s"],
                                "sharded_symmetric_ms": cd_sharded["symmetric_dealt"]["ms"],
                                "sharded_symmetric_form": "every unordered tile pair once in the whole job, row blocks dealt round-robin "
                                                          "(BSG_CD_DEAL), per-aircraft outputs all-reduced; identical conflicts"})
        line = {"metric": "env_steps_per_sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
                "warmup": W, "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 (lat/lon f64)", "data": "synthetic", "config": workload_config(world),
                "value_l2_warm": warm_value, "e2e": e2e, "gpu_launches": launches, "cd_pairs_headline": cd_head,
                "baseline_configs": legs, "roofline": roof,
                "cpu_baseline": cb, "clocks": clk.summary(), "cd_pairs": cd}
        if other is not None:
            line["other_envs"] = other
        if traffic_leg is not None:
            line["airspace_traffic"] = traffic_leg
        if cd_sharded is not None:
            line["cd_pairs_sharded"] = cd_sharded
        if traffic_sharded is not None:
            line["airspace_traffic_sharded"] = traffic_sharded
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if line is not None:
        print(json.dumps(line), file=_OUT, flush=True)


def step_outputs(obs, reward, terminated, truncated):
    """Host float32 copies of what BlueSkyVectorEnv.step_torch returned, by --dump-outputs file name (E x 103 obs values
    + 3 x E: 1.7 MB at 4096 envs)."""
    arrays = {"obs_" + k: v for k, v in obs.items()}
    arrays.update(reward=reward, terminated=terminated, truncated=truncated)
    return {k: v.float().cpu().numpy() for k, v in arrays.items()}


def bench_env_leg(torch, dev, BlueSkyVectorEnv, env_id, E, kw, world, rank, max_over_ranks, barrier, steps=60):
    """Device time per batched step of one env configuration, E envs on EVERY rank (weak scaling, global env ids), L2
    flushed between steps, max over ranks; returns whole-job env-steps/s."""
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    v = BlueSkyVectorEnv(env_id, E, device=dev.index, seed=0, autoreset_mode="same_step", env_id_offset=rank * E, **kw)
    v.reset_torch()
    g = torch.Generator(device=dev).manual_seed(77 + rank)
    a = torch.rand((steps + 5, E, v.layout.act_dim), device=dev, generator=g) * 2.0 - 1.0
    for i in range(PREROLL_STEPS + 5):                     # (stationary regime first, as in the headline loop)
        v.step_torch(a[i % (steps + 5)])
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    torch.cuda._sleep(int(steps * 60e-6 * 1.9e9))          # (head start for the host, as in the headline loop)
    for i in range(steps):
        flush.fill_(float(i))
        ev[i][0].record()
        v.step_torch(a[5 + i])
        ev[i][1].record()
    barrier()
    t = max_over_ranks(sum(x.elapsed_time(y) for x, y in ev) * 1e-3)
    v.close()
    return {"envs_per_gpu": E, "envs_total": E * world, "ms_per_step": 1e3 * t / steps, "env_steps_per_s": E * world * steps / t}


# BASELINE configs[2] and [3] (run at every N), then context-only variants (single GPU)
CONFIG_LEGS = (("configs[2] SectorCREnv-v0, 8192 envs per GPU (65 536 over 8), CD on", "SectorCREnv-v0", 8192, dict(cd_enabled=True)),
               ("configs[3] MergeEnv-v0, 4096 envs per GPU, FMS-guided intruders, CD on", "MergeEnv-v0", 4096, dict(cd_enabled=True)))
CONTEXT_LEGS = (("HorizontalCREnv-v0 configs[1] at 3000 m instead of the reference's 0 m (SURVEY 8d variant)", "HorizontalCREnv-v0", 4096,
                 dict(cd_enabled=True, n_intruders=20, init_alt=3000.0)),
                ("DescentEnv-v0 (configs[0], batched)", "DescentEnv-v0", 65536, {}),
                ("HorizontalCREnv-v0 reference default (5 intruders, no CD)", "HorizontalCREnv-v0", 65536, {}))


def C_double_probe(lib, device):
    import ctypes as C
    from bluesky_gym_sasha_b200 import _lib
    out = C.c_double(0.0)
    _lib.check(lib.bsg_probe_fp32(device, C.byref(out)))
    return out.value


def bench_cd(torch, dev, StateBasedCD, fp32_peak, n=CD_N, reps=5):
    """All-pairs CD at N = 100k on one GPU: ordered pairs/s and fraction of the measured FP32 peak."""
    rng = np.random.default_rng(1)
    lat = 52 + 40 * (rng.random(n) - 0.5)
    lon = 4 + 40 * (rng.random(n) - 0.5)
    alt = np.round(rng.uniform(3000, 12000, n) / 304.8) * 304.8
    gs = rng.uniform(150, 250, n)
    trk = rng.uniform(0, 360, n)
    vs = np.where(rng.random(n) < 0.8, 0.0, rng.choice([-1.0, 1.0], n) * rng.uniform(5, 15, n))
    cd = StateBasedCD(device=dev.index)
    rec, _ = cd.pack(lat, lon, trk, gs, alt, vs, 52.0, 4.0)
    for _ in range(2):
        out = cd.detect_packed(rec, n)
    torch.cuda.synchronize(dev)
    best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = cd.detect_packed(rec, n)
        e1.record()
        torch.cuda.synchronize(dev)
        best = min(best, e0.elapsed_time(e1) * 1e-3)
    pairs = n * (n - 1)
    tf = pairs * F_PAIR / best / 1e12
    res = {"n_aircraft": n, "ordered_pairs_per_s": pairs / best, "ms": best * 1e3, "n_conf": int(out["npairs"][0]),
           "n_los": int(out["npairs"][1]),
           "roofline": {"bound": "fp32", "achieved": tf, "peak": fp32_peak / 1e12, "unit": "TFLOP/s",
                        "frac": tf / (fp32_peak / 1e12), "flop_per_pair": F_PAIR, "executed_fraction": 1.0,
                        "kernel": "cd_tiled_kernel"}}
    # same detection with spatial culling (identical conflict sets; the brute-force figure above is the headline)
    d = [cd._as_dev(x) for x in (lat, lon, trk, gs, alt, vs)]
    prep = 1e30
    for _ in range(4):                      # spatial order + pack on the device (bsg_cd_pack_ordered: grid binning, counting sort)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rec_s, _, perm = cd.pack_ordered(*d, 52.0, 4.0)
        e1.record()
        torch.cuda.synchronize(dev)
        prep = min(prep, e0.elapsed_time(e1) * 1e-3)
    for _ in range(2):
        outc = cd.detect_packed(rec_s, n, cull=True)
    torch.cuda.synchronize(dev)
    bestc = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        outc = cd.detect_packed(rec_s, n, cull=True)
        e1.record()
        torch.cuda.synchronize(dev)
        bestc = min(bestc, e0.elapsed_time(e1) * 1e-3)
    n_tiles = (n + 255) // 256
    off = 16 * ((n_tiles * 12 * 4 + 15) // 16)
    kept = int(cd._buf["cull_work"][off:off + 4 * n_tiles].view(torch.int32).sum())
    for name, kw in (("symmetric", dict(symmetric=True)), ("culled_symmetric", dict(symmetric=True, cull=True))):
        for _ in range(2):
            outs = cd.detect_packed(rec_s, n, **kw)
        torch.cuda.synchronize(dev)
        bests = 1e30
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            outs = cd.detect_packed(rec_s, n, **kw)
            e1.record()
            torch.cuda.synchronize(dev)
            bests = min(bests, e0.elapsed_time(e1) * 1e-3)
        res[name] = {"ordered_pairs_per_s": pairs / bests, "ms": bests * 1e3, "n_conf": int(outs["npairs"][0]),
                     "n_los": int(outs["npairs"][1]),
                     "note": "BSG_CD_SYMMETRIC: every unordered tile pair once, both ordered results emitted (executed fraction ~0.5"
                             + (" of the culled tile pairs)" if "cull" in kw else ")")}
    res["forms_agree"] = all(res[k]["n_conf"] == res["n_conf"] and res[k]["n_los"] == res["n_los"] for k in ("symmetric", "culled_symmetric")) \
        and int(outc["npairs"][0]) == res["n_conf"] and int(outc["npairs"][1]) == res["n_los"]
    res["culled"] = {"ordered_pairs_per_s": pairs / bestc, "ms": bestc * 1e3, "ms_sort_and_pack": prep * 1e3,
                     "ms_incl_sort_and_pack": bestc * 1e3 + prep * 1e3,
                     "ordered_pairs_per_s_incl_sort_and_pack": pairs / (bestc + prep),
                     "executed_fraction": kept / float(n_tiles * n_tiles), "n_conf": int(outc["npairs"][0]),
                     "n_los": int(outc["npairs"][1]),
                     "note": "bsg_cd_detect_culled on records in the device-chosen spatial order (bsg_cd_pack_ordered: grid binning + counting sort + pack, no library sort): tile pairs out of reach (rpz + (v_a+v_b)*300 s) skipped"}
    return res


def bench_traffic(torch, dev, hbm_peak, n=CD_N, reps=20):
    """SURVEY 8f-4 leg: one airspace of n aircraft (the C5 box) flying four-waypoint routes with altitude constraints under
    VNAV, state-based detection every substep (culled + symmetric K2 with pair lists) and MVP resolution: device time per
    simulator substep and of bsg_traf_substep alone (HBM-bound: 328 algorithmic bytes per aircraft-substep)."""
    import ctypes as C
    from bluesky_gym_sasha_b200 import _lib
    from bluesky_gym_sasha_b200.cd import StateBasedCD, _ptr
    from bluesky_gym_sasha_b200.traffic import AirspaceTraffic
    rng = np.random.default_rng(3)
    lat, lon = 52 + 40 * (rng.random(n) - 0.5), 4 + 40 * (rng.random(n) - 0.5)
    perm = StateBasedCD.spatial_order(torch.as_tensor(lat, device=dev), torch.as_tensor(lon, device=dev)).cpu().numpy()
    lat, lon = lat[perm], lon[perm]                    # created in spatially coherent order: the culled detection needs it
    alt = np.round(rng.uniform(3000, 12000, n) / 304.8) * 304.8
    hdg, cas = rng.uniform(0, 360, n), rng.uniform(120, 150, n)
    W = 4
    wlat, wlon, walt = np.zeros((n, W)), np.zeros((n, W)), np.full((n, W), -999.0)
    la, lo, brg = lat.copy(), lon.copy(), hdg.copy()
    for k in range(W):
        d = rng.uniform(60.0, 120.0, n) / 111.0
        la = la + d * np.cos(np.radians(brg)); lo = lo + d * np.sin(np.radians(brg)) / np.cos(np.radians(np.clip(la, -80, 80)))
        brg = brg + rng.uniform(-40, 40, n)
        wlat[:, k], wlon[:, k] = la, lo
        walt[:, k] = np.where(rng.random(n) < 0.5, np.clip(alt + rng.uniform(-2500, 1500, n), 1500, 12000), -999.0)
    tr = AirspaceTraffic(n, device=dev.index, simdt=1.0, reso="MVP", reso_mode=1, max_wpts=W)
    tr.create(lat, lon, hdg, alt, cas)
    tr.set_routes(np.arange(n), wlat, wlon, walt, None)
    tr.step(20)                                         # warm-up (first resolutions, VNAV profiles computed)
    torch.cuda.synchronize(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * reps)]
    for r in range(reps):
        ev[2 * r].record(); tr.step(1); ev[2 * r + 1].record()
    torch.cuda.synchronize(dev)
    t_sub = sorted(ev[2 * r].elapsed_time(ev[2 * r + 1]) for r in range(reps))[reps // 2]
    # the fused per-aircraft kernel alone, on the state and conflict list of the last substep
    out = tr.last
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)
    cfg0 = _lib.TrafConfig.from_buffer_copy(tr.cfg)
    cfg0.reso = 0                                       # the per-aircraft kernel alone would need the index of this list:
    ts, ts_all = [], []                                 # timed (a) without ASAS and (b) as the whole call (index + kernel)
    for r in range(2 * reps):
        flush.fill_(float(r))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        _lib.check(tr.lib.bsg_traf_substep(C.byref(tr.cfg if r % 2 else cfg0), C.byref(tr.tt), _ptr(tr.rec), 0, _ptr(out["pairs"]),
                                           _ptr(out["attr"]), _ptr(out["npairs"]), None, tr.cd.pair_capacity, _ptr(tr.work),
                                           tr.work.numel(), st))
        b.record()
        torch.cuda.synchronize(dev)
        (ts_all if r % 2 else ts).append(a.elapsed_time(b))
    t_k, t_call = sorted(ts)[reps // 2], sorted(ts_all)[reps // 2]
    nconf, nlos = (int(v) for v in out["npairs"].cpu())
    bytes_per_ac = 328
    # the same kernel where its bound shows: 2^20 aircraft (344 MB of state, larger than L2), detection off
    big = 1 << 20
    tb = AirspaceTraffic(big, device=dev.index, simdt=1.0, max_wpts=W, pair_capacity=4096)
    reps_b = -(-big // n)
    tile = lambda a: np.tile(a, (reps_b,) + (1,) * (a.ndim - 1))[:big]
    tb.create(tile(lat), tile(lon), tile(hdg), tile(alt), tile(cas))
    tb.set_routes(np.arange(big), tile(wlat), tile(wlon), tile(walt), None)
    tb.step(3, detect=False)
    tsb = []
    for r in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); tb.step(1, detect=False); b.record()
        torch.cuda.synchronize(dev)
        tsb.append(a.elapsed_time(b))
    t_big = sorted(tsb)[reps // 2]
    del tb
    return {"n_aircraft": n, "ms_per_substep": t_sub, "aircraft_substeps_per_s": n / (t_sub * 1e-3),
            "realtime_factor": 1.0 / (t_sub * 1e-3), "n_conf": nconf, "n_los": nlos, "counters": tr.counters(),
            "form": "bsg_traf_pack + culled symmetric K2 with pair lists + bsg_traf_substep (conflict index + fused per-aircraft kernel), MVP horizontal, VNAV routes",
            "substep_call_us": t_call * 1e3,
            "substep_kernel": {"us": t_k * 1e3, "l2": "flushed", "what": "traf_substep_kernel with reso off (autopilot / VNAV / limits / kinematics)", "roofline": {
                "bound": "hbm", "achieved": bytes_per_ac * n / (t_k * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": bytes_per_ac * n / (t_k * 1e-3) / 1e9 / hbm_peak, "bytes_per_aircraft_substep": bytes_per_ac,
                "kernel": "traf_substep_kernel"}},
            "substep_kernel_2e20_aircraft": {"us": t_big * 1e3, "l2": "state (344 MB) exceeds L2", "roofline": {
                "bound": "hbm", "achieved": bytes_per_ac * big / (t_big * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": bytes_per_ac * big / (t_big * 1e-3) / 1e9 / hbm_peak, "kernel": "traf_substep_kernel"}}}


def bench_traffic_sharded(torch, dist, dev, world, rank, max_over_ranks, barrier, n=CD_N, reps=20):
    """bench_traffic's airspace (N aircraft, four-waypoint VNAV routes, MVP) with the aircraft block-partitioned over the
    ranks (AirspaceTraffic(group=True)): per substep every rank packs its block, the records are all-gathered over NVLink,
    each rank detects its own rows against the whole airspace (culled form, pair lists) and advances its own aircraft.
    Device time per substep, max over ranks."""
    from bluesky_gym_sasha_b200.cd import StateBasedCD
    from bluesky_gym_sasha_b200.traffic import AirspaceTraffic
    rng = np.random.default_rng(3)
    lat, lon = 52 + 40 * (rng.random(n) - 0.5), 4 + 40 * (rng.random(n) - 0.5)
    perm = StateBasedCD.spatial_order(torch.as_tensor(lat, device=dev), torch.as_tensor(lon, device=dev)).cpu().numpy()
    lat, lon = lat[perm], lon[perm]
    alt = np.round(rng.uniform(3000, 12000, n) / 304.8) * 304.8
    hdg, cas = rng.uniform(0, 360, n), rng.uniform(120, 150, n)
    W = 4
    wlat, wlon, walt = np.zeros((n, W)), np.zeros((n, W)), np.full((n, W), -999.0)
    la, lo, brg = lat.copy(), lon.copy(), hdg.copy()
    for k in range(W):
        d = rng.uniform(60.0, 120.0, n) / 111.0
        la = la + d * np.cos(np.radians(brg)); lo = lo + d * np.sin(np.radians(brg)) / np.cos(np.radians(np.clip(la, -80, 80)))
        brg = brg + rng.uniform(-40, 40, n)
        wlat[:, k], wlon[:, k] = la, lo
        walt[:, k] = np.where(rng.random(n) < 0.5, np.clip(alt + rng.uniform(-2500, 1500, n), 1500, 12000), -999.0)
    per = -(-(-(-n // world)) // 256) * 256
    sl = slice(min(rank * per, n), min((rank + 1) * per, n))
    tr = AirspaceTraffic(per, device=dev.index, simdt=1.0, reso="MVP", reso_mode=1, max_wpts=W, group=True)
    if sl.stop > sl.start:
        tr.create(lat[sl], lon[sl], hdg[sl], alt[sl], cas[sl])
        tr.set_routes(np.arange(sl.stop - sl.start), wlat[sl], wlon[sl], walt[sl], None)
    tr.step(20)
    barrier()
    best = 1e30
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        tr.step(reps)
        e1.record()
        torch.cuda.synchronize(dev)
        best = min(best, max_over_ranks(e0.elapsed_time(e1) / reps))
    nconf = torch.tensor([int(tr.last["npairs"][0])], dtype=torch.int64, device=dev)
    dist.all_reduce(nconf)
    return {"n_aircraft": n, "aircraft_per_gpu": per, "ms_per_substep": best, "aircraft_substeps_per_s": n / (best * 1e-3),
            "realtime_factor": 1.0 / (best * 1e-3), "n_conf": int(nconf.item()),
            "form": "per substep: bsg_traf_pack of the own block, ncclAllGather of the 32 B records, culled K2 of the own rows "
                    "against the whole airspace with pair lists, all-reduce of the conflict count, bsg_traf_substep of the own "
                    "aircraft (MVP horizontal, VNAV routes); results identical to the unsharded airspace (scripts/traf_sharded_check.py)"}


def bench_cd_sharded(torch, dist, dev, StateBasedCD, world, rank, max_over_ranks, barrier, n=CD_N, reps=5):
    """N = 100k aircraft block-partitioned over the ranks: pack own block, all-gather the 32 B records over
    NVLink, evaluate own rows against all columns.  Time = max over ranks of (all-gather + detection)."""
    per = -(-n // world)
    per = -(-per // 256) * 256                      # tile-aligned blocks
    n_tot = per * world
    rng = np.random.default_rng(1)
    lat = 52 + 40 * (rng.random(n_tot) - 0.5)
    lon = 4 + 40 * (rng.random(n_tot) - 0.5)
    alt = np.round(rng.uniform(3000, 12000, n_tot) / 304.8) * 304.8
    gs = rng.uniform(150, 250, n_tot)
    trk = rng.uniform(0, 360, n_tot)
    vs = np.where(rng.random(n_tot) < 0.8, 0.0, rng.choice([-1.0, 1.0], n_tot) * rng.uniform(5, 15, n_tot))
    sl = slice(rank * per, (rank + 1) * per)
    cd = StateBasedCD(device=dev.index)
    align = torch.zeros(1, device=dev)
    rec, _ = cd.pack(lat[sl], lon[sl], trk[sl], gs[sl], alt[sl], vs[sl], 52.0, 4.0)
    for _ in range(2):
        out = cd.detect_sharded(rec, per, want_pairs=True)
    barrier()
    best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        dist.all_reduce(align)         # (device-side: the ranks' streams reach e0 together, whatever the hosts' skew after the barrier)
        e0.record()
        out = cd.detect_sharded(rec, per, want_pairs=True)
        e1.record()
        torch.cuda.synchronize(dev)
        best = min(best, max_over_ranks(e0.elapsed_time(e1) * 1e-3))
    nconf = torch.tensor([int(out["npairs"][0])], dtype=torch.int64, device=dev)
    dist.all_reduce(nconf)
    res = {"n_aircraft": n_tot, "rows_per_gpu": per, "ordered_pairs_per_s": n_tot * (n_tot - 1) / best, "ms": best * 1e3,
           "n_conf": int(nconf.item()), "collective": "ncclAllGather of 32 B records, then row-sharded tiles"}
    # culled form: the aircraft are dealt to the ranks in the global strip-sorted order (identical conflict sets)
    d = [cd._as_dev(x) for x in (lat, lon, trk, gs, alt, vs)]
    perm = cd.spatial_order(d[0], d[1])[sl.start:sl.stop]
    rec_s, _ = cd.pack(*[x[perm] for x in d], 52.0, 4.0)
    for _ in range(2):
        outc = cd.detect_sharded(rec_s, per, cull=True, want_pairs=True)
    barrier()
    bestc = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        dist.all_reduce(align)         # (device-side: the ranks' streams reach e0 together, whatever the hosts' skew after the barrier)
        e0.record()
        outc = cd.detect_sharded(rec_s, per, cull=True, want_pairs=True)
        e1.record()
        torch.cuda.synchronize(dev)
        bestc = min(bestc, max_over_ranks(e0.elapsed_time(e1) * 1e-3))
    nconfc = torch.tensor([int(outc["npairs"][0])], dtype=torch.int64, device=dev)
    dist.all_reduce(nconfc)
    res["culled"] = {"ordered_pairs_per_s": n_tot * (n_tot - 1) / bestc, "ms": bestc * 1e3, "n_conf": int(nconfc.item())}
    # symmetric forms with the row blocks dealt round-robin to the ranks (BSG_CD_DEAL): every unordered tile pair once in
    # the whole job, per-aircraft outputs all-reduced (time incl. the gather and the three all-reduces)
    for name, r, cull in (("symmetric_dealt", rec, False), ("culled_symmetric_dealt", rec_s, True)):
        for _ in range(2):
            outd = cd.detect_sharded_symmetric(r, per, cull=cull)
        barrier()
        bestd = 1e30
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            dist.all_reduce(align)
            e0.record()
            outd = cd.detect_sharded_symmetric(r, per, cull=cull)
            e1.record()
            torch.cuda.synchronize(dev)
            bestd = min(bestd, max_over_ranks(e0.elapsed_time(e1) * 1e-3))
        res[name] = {"ordered_pairs_per_s": n_tot * (n_tot - 1) / bestd, "ms": bestd * 1e3, "n_conf": int(outd["npairs"][0]),
                     "collective": "ncclAllGather of the records, all-reduce of the per-aircraft counts / tcpamax / totals"}
    # no-gather forms: column tiles read from the owning GPU over NVLink inside the CD kernel (bsg_cd_detect_peers)
    try:
        for name, r, cull in (("p2p", rec, False), ("p2p_culled", rec_s, True)):
            for _ in range(2):
                outp = cd.detect_sharded_p2p(r, per, cull=cull, want_pairs=True)
            barrier()
            bestp = 1e30
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                barrier()
                dist.all_reduce(align)
                e0.record()
                outp = cd.detect_sharded_p2p(r, per, cull=cull, want_pairs=True)
                e1.record()
                torch.cuda.synchronize(dev)
                bestp = min(bestp, max_over_ranks(e0.elapsed_time(e1) * 1e-3))
            nc = torch.tensor([int(outp["npairs"][0])], dtype=torch.int64, device=dev)
            dist.all_reduce(nc)
            res[name] = {"ordered_pairs_per_s": n_tot * (n_tot - 1) / bestp, "ms": bestp * 1e3, "n_conf": int(nc.item()),
                         "collective": "none on the data path: TMA loads of peer tiles over NVLink (symmetric memory)"}
    except Exception as ex:                      # symmetric memory unavailable on this box: report, do not fail the bench
        res["p2p"] = {"unavailable": repr(ex)[:200]}
    # every form must find the same conflicts
    res["forms_agree"] = all(v.get("n_conf", res["n_conf"]) == res["n_conf"] for v in res.values() if isinstance(v, dict))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--skip-cpu", action="store_true", help="omit the cpu_baseline leg (profiling runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 step path")
    # The contract is ONE JSON line on stdout.  Libraries write banners to fd 1 from native code (NCCL prints its version
    # there when NCCL_DEBUG asks for it), so fd 1 points at stderr while the bench runs and the line goes to the saved fd.
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
    _OUT.flush()


if __name__ == "__main__":
    main()
