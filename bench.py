#!/usr/bin/env python
"""bench.py -- B747 env-steps/s on 1..8 B200 next to the reference CPU path.

Workload (BASELINE.json configs[2], the configuration the metric is quoted on): 1 Mi environments per
GPU, fp32 mode, K = 10 fused RK4 substeps per env step, in-kernel auto-reset, canonical env
configuration (PID_LIKE obs, CLASSIC reward, MANUAL / DIRECT_CONTROL, CONST reference, tk = 20 s).
A "step" is one env step of every environment = one kernel launch per GPU.  Environments are
partitioned across ranks (weak scaling, no collective on the step path; only the episode statistics
are reduced once, after the timed region).

  python bench.py [--gpus N] [--steps K] [--warmup W]        # this repo's CUDA path
  python bench.py ... --dump-outputs DIR                     # + obs / reward / done of the last timed step as .npy
  python bench.py --impl reference ...                       # the reference DLL on the host cores
Under torchrun (N > 1) one rank per GPU; rank 0 prints ONE JSON line.
"""
import argparse
import atexit
import json
import math
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ENVS_PER_GPU = 1 << 20
SUBSTEPS = 10
METRIC = "B747 env-steps/sec"
UNIT = "env-steps/s"
WORKLOAD = ("1Mi envs/GPU, fp32 mode, K=10 fused RK4 substeps, in-kernel auto-reset, canonical env "
            "(PID_LIKE obs, CLASSIC reward, MANUAL/DIRECT_CONTROL, CONST ref, tk=20)")
# algorithmic HBM bytes per env step of the f32 LEAN layout (b747_kernels_f32.cu): 9 x 16-byte state
# groups in + out, action 4, obs 12, reward 4, done 1
BYTES_PER_ENV_STEP = 2 * 9 * 16 + 4 + 12 + 4 + 1


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)  # no sampler outlives the benchmark, even when a step raises
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mxc = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx = mxc
            if t0 - 0.05 <= t <= t1 + 0.05:
                sm.append(clk)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # region shorter than the sampling period: use the nearest samples
            sm = [float(r[1].split(",")[1]) for r in self.rows[-3:] if len(r[1].split(",")) > 2]
        sm.sort()
        return {"sm_mhz": (sm[len(sm) // 2] if sm else None), "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# reference arm: the reference DLL's own machine code (oracle/_ref) driven by the oracle's C env layer,
# one private DLL instance per worker process, all host cores.
# ------------------------------------------------------------------------------------------------
def _ref_worker(args):
    wid, n_steps, substeps, repeats = args
    import numpy as np
    from oracle import oracle as O
    from oracle import dllref
    cfg = O.make_cfg(sample_time=substeps * 0.01, seed=1)
    if dllref.available():
        env = O.RefEnv(cfg, env_id=wid)
        env.reset()
        dllref.sandbox()  # this worker only computes from here on: no sockets, exec, ptrace or file writes (seccomp)
        run = lambda a: env.rollout(a, auto_reset=True, record=False)
    else:
        ob = O.OracleBatch(cfg, 1, env_id_offset=wid)
        ob.reset()

        def run(a):
            for x in a:
                ob.step([x])
    rng = np.random.default_rng(wid)
    acts = rng.uniform(-1, 1, n_steps)
    times = []
    for _ in range(repeats):
        t = time.perf_counter()
        run(acts)
        times.append(time.perf_counter() - t)
    return times


def cpu_reference_rate(steps, warmup, env_steps_per_worker, substeps=SUBSTEPS):
    """env-steps/s of the reference CPU path with every host core busy; returns (value, info)."""
    from oracle import dllref
    from oracle import oracle as O
    O.build()
    cores = os.cpu_count() or 1
    kind = "reference" if dllref.available() else "port"
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        res = pool.map(_ref_worker, [(w, env_steps_per_worker, substeps, warmup + steps) for w in range(cores)])
    # per-repeat wall time = slowest worker; every repeat processes cores * env_steps_per_worker env steps
    per_rep = [max(r[i] for r in res) for i in range(warmup, warmup + steps)]
    total = sum(per_rep)
    value = cores * env_steps_per_worker * steps / total
    sample = (f"{cores} workers x {env_steps_per_worker} env-steps x {steps} timed repeats, K={substeps}, canonical env, "
              + ("reference DLL machine code (oracle/_ref) + C env layer" if kind == "reference"
                 else "oracle C restatement (oracle/_ref not built)"))
    return value, {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample}, total / steps


def python_loop_rate(n_steps=20000, substeps=SUBSTEPS):
    """SURVEY.md 8d (ii): a gym-style Python loop, one `env.step(a)` call per env step on the DLL-backed env layer, one
    core.  An upper bound for any Python-side ControllerEnv (the reference's wrappers add ~50 ctypes property accesses
    per step; its published end-to-end figure is 240-360 env-steps/s)."""
    import numpy as np
    from oracle import dllref
    from oracle import oracle as O
    if not dllref.available():
        return None
    env = O.RefEnv(O.make_cfg(sample_time=substeps * 0.01, seed=1), env_id=0)
    env.reset()
    acts = np.random.default_rng(0).uniform(-1, 1, n_steps)
    t = time.perf_counter()
    for a in acts:
        _, _, d = env.step(a)
        if d:
            env.reset()
    dt = time.perf_counter() - t
    return {"value": n_steps / dt, "unit": UNIT, "cores": 1,
            "sample": f"{n_steps} env.step(a) calls from a Python loop, K={substeps}, reference DLL + C env layer"}


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path (its DLL's machine code + the C env layer) on every host core;
    each step is a bounded sample of the arm's workload: 20000 env-steps per worker."""
    if rank != 0:
        return
    K = CONFIGS[args.config][3]
    value, info, sec_per_step = cpu_reference_rate(args.steps, args.warmup, 20000, substeps=K)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": _config_dict(args.config),
            "cpu_baseline": info,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


def _bind_near_gpu(torch, local_rank):
    """Run this rank (and first-touch its pinned buffers) on the CPUs NVML reports as local to its GPU: with 8 ranks
    the host legs of the e2e path otherwise cross sockets.  Best effort; returns a short description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        p = torch.cuda.get_device_properties(local_rank)
        bus = "%08x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (max(ncpu, 1024) + 63) // 64)
        allowed = os.sched_getaffinity(0)
        cpus = {i for i in allowed if (words[i // 64] >> (i % 64)) & 1}
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} of {len(allowed)} cpus (GPU-local)"
        return f"{len(allowed)} cpus (no narrower GPU-local set)"
    except Exception as e:  # NVML missing / restricted: keep the default affinity
        return f"default ({type(e).__name__})"


# ------------------------------------------------------------------------------------------------
CONFIGS = {
    # name: (engine kwargs, envs per GPU, dtype name, substeps, workload string, algorithmic bytes per env step)
    "fp32_1M_K10": (dict(), N_ENVS_PER_GPU, "f32", SUBSTEPS, WORKLOAD, BYTES_PER_ENV_STEP),
    # BASELINE configs[1]: the float64 parity mode (DLL operation order, -fmad=false), K = 5 (main.py's sample_time)
    "fp64_4096": (dict(), 4096, "f64", 5,
                  "4096 envs, fp64 parity mode (DLL operation order), K=5, in-kernel auto-reset, canonical env", None),
    "fp64_256k": (dict(), 1 << 18, "f64", 10,
                  "256Ki envs, fp64 parity mode (DLL operation order), K=10, in-kernel auto-reset, canonical env", None),
    # the general layout with the altitude loop (ResetRefMode.HYBRID, swept by main.py:89-94): kernel tier 2
    "tier2_1M_K10": (dict(reset_ref_mode=2), N_ENVS_PER_GPU, "f32", SUBSTEPS,
                     "1Mi envs/GPU, fp32 mode, K=10, HYBRID reset (altitude loop in half of the episodes), PID_LIKE obs, "
                     "CLASSIC reward", None),
}
# float64 handle: 45 state slots in + out, tick / flags / episode words in + out, action, 3 obs, reward, done
BYTES_F64 = 2 * 45 * 8 + 2 * 12 + 8 + 24 + 8 + 1
# general f32 layout with the altitude loop (tier 2): D groups 0-10 + F groups 0-4 in, D 0-7 + F 0-2,4 out
BYTES_TIER2 = (11 + 5) * 16 + (8 + 4) * 16 + 4 + 12 + 4 + 1


def _config_dict(name):
    """`config` of the JSON line -- identical for the CUDA arm and the reference arm (same workload definition)."""
    kw, n_local, dtype_name, K, workload, bytes_env = CONFIGS[name]
    if bytes_env is None:
        bytes_env = BYTES_F64 if dtype_name == "f64" else BYTES_TIER2
    ep_len = int(round(20.0 / (K * 0.01)))
    return {"workload": workload, "envs_per_gpu": n_local, "substeps": K,
            "episode_phases": f"spread uniformly over the {ep_len}-step episode before the timed region "
                              f"(~1/{ep_len} of the envs auto-reset in every step)",
            "l2": f"per-launch working set {bytes_env * n_local / 1e6:.0f} MB of env state"
                  + (" > 126 MB L2 (no flush needed)" if bytes_env * n_local > 126e6 else
                     " < 126 MB L2: state stays L2-resident between launches, as it does in use")}


def _desync(eng, torch, n, ep_len, pool, obs, rew, done, dev):
    """Spread the episode phases uniformly (a VecEnv whose envs all start together stays in lock-step for ever: every
    episode lasts exactly tk / sample_time steps): after `ep_len` steps with a masked reset of the envs
    id % ep_len == t at step t, 1 / ep_len of the envs finishes in every later launch -- the steady state of a
    rollout with in-kernel auto-reset (Philox draws, full-group stores, ballot + shuffles + atomics all in the timed
    region)."""
    ids = torch.arange(n, device=dev)
    for t in range(ep_len):
        eng.step(pool[t % len(pool)], obs, rew, done)
        eng.reset(mask=((ids % ep_len) == t).to(torch.uint8))
    eng.step(pool[0], obs, rew, done)
    eng.synchronize()
    eng.episode_stats()  # the warm-up episodes do not count


def run_cuda(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist
    from b747_rl_ctrl_b200 import engine as E
    from b747_rl_ctrl_b200.sharding import reduce_episode_stats, shard_range, summarize

    kw, n_local, dtype_name, K, workload, bytes_env = CONFIGS[args.config]
    main_cfg = args.config == "fp32_1M_K10"
    dtype = E.F32 if dtype_name == "f32" else E.F64
    if bytes_env is None:
        bytes_env = BYTES_F64 if dtype == E.F64 else BYTES_TIER2
    tdt = torch.float32 if dtype == E.F32 else torch.float64
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    affinity = _bind_near_gpu(torch, local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n_total = n_local * world
    lo, hi = shard_range(n_total, world, rank)
    ep_len = int(round(20.0 / (K * 0.01)))

    def make_engine():
        e = E.BatchEngine(n_envs=hi - lo, dtype=dtype, device=local_rank, sample_time=K * 0.01, seed=1,
                          env_id_offset=lo, auto_reset=True, **kw)
        e.use_stream(torch.cuda.current_stream().cuda_stream)  # torch's stream: torch.cuda.Event brackets the kernels
        return e

    eng = make_engine()
    act, obs, rew, done = eng.alloc_io()
    eng.reset(obs)
    # synthetic action stream: a pool of pre-generated U(-1,1) arrays, resident in HBM
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    pool = [torch.empty(n_local, device=dev, dtype=tdt).uniform_(-1, 1, generator=gen) for _ in range(8)]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_pass(e, steps):
        """EXACTLY `steps` steps bracketed by barrier + synchronize; returns (ms total, per-launch ms list)."""
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        barrier()
        ev[0].record()
        for i in range(steps):
            e.step(pool[i % 8], obs, rew, done)
            ev[i + 1].record()
        barrier()
        return ev[0].elapsed_time(ev[-1]), [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]

    warm = max(args.warmup, 3)
    # ---- lock-step phases first (a fresh handle: every env in the same flight phase, no env finishes in the window)
    for i in range(warm):
        eng.step(pool[i % 8], obs, rew, done)
    lock_ms, _ = timed_pass(eng, min(args.steps, 100))
    lock_steps = min(args.steps, 100)
    # ---- steady state: episode phases spread uniformly, ~1/ep_len of the envs auto-reset in every launch
    _desync(eng, torch, n_local, ep_len, pool, obs, rew, done, dev)
    for i in range(warm):
        eng.step(pool[i % 8], obs, rew, done)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    launches0 = eng.launch_count
    t_wall0 = time.time()
    ms_total, per_launch_ms = timed_pass(eng, args.steps)        # THE timed region: exactly args.steps steps
    # what the last timed step handed back, copied before the repeats below step the envs further
    dumped = {"obs": obs.cpu(), "reward": rew.cpu(), "done": done.cpu()} if args.dump_outputs and rank == 0 else None
    launches = eng.launch_count - launches0
    stats_timed = eng.episode_stats()                              # episodes finished inside the timed region
    # clock samples need >= 0.5 s under load (nvidia-smi samples every 100 ms; 20 steps last 6 ms): the same timed pass is
    # repeated, the sampler keeps running across the timed region and the repeats, the repeats' spread is reported
    rep_ms = [ms_total / args.steps]
    # the number of repeats is derived from the max-over-ranks time of the first pass, so every rank runs the SAME number
    # of barriers (a per-rank wall-clock loop dead-locks the ranks against each other)
    t_first = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_first, op=dist.ReduceOp.MAX)
    n_rep = int(min(500, max(1, math.ceil(700.0 / max(float(t_first.item()), 1e-3)))))
    for _ in range(n_rep):
        m, _ = timed_pass(eng, args.steps)
        rep_ms.append(m / args.steps)
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    t = torch.tensor([ms_total, lock_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total_max, lock_ms_max = float(t[0].item()), float(t[1].item())
    value = n_total * args.steps / (ms_total_max * 1e-3)
    eng.episode_stats()

    # ---- end-to-end through the public host API: pinned host buffers, H2D + D2H inside the timed region
    e2e = None
    e2e_steps = max(3, min(args.steps, 30))
    if dtype == E.F32 and eng.obs_dim == 3:
        # b747_step_host_packed: the kernel reads the actions from and stores (obs[3], reward) records into the pinned
        # host buffers directly (zero-copy over PCIe), the done bits come back with one small copy
        h_act = [torch.empty(n_local, dtype=torch.float32).uniform_(-1, 1).pin_memory() for _ in range(4)]
        h_out = torch.empty(n_local, 4, dtype=torch.float32).pin_memory()
        h_bits = torch.empty((n_local + 31) // 32, dtype=torch.int32).pin_memory()
        step_e2e = lambda i: eng.step_host_packed(h_act[i % 4].numpy(), h_out.numpy(), h_bits.numpy())
        d2h = 16 * n_local + 4 * ((n_local + 31) // 32)
        api = ("b747_step_host_packed (C ABI, pinned host buffers): one launch, actions read and (obs[3], reward) records "
               "stored zero-copy over PCIe by the kernel, done flags as one bit per env copied back")
    else:
        es = 4 if dtype == E.F32 else 8
        npd = np.float32 if dtype == E.F32 else np.float64
        h_act = [torch.empty(n_local, dtype=tdt).uniform_(-1, 1).pin_memory() for _ in range(4)]
        h_obs = torch.empty(n_local, eng.obs_dim, dtype=tdt).pin_memory()
        h_rew = torch.empty(n_local, dtype=tdt).pin_memory()
        h_done = torch.empty(n_local, dtype=torch.uint8).pin_memory()
        step_e2e = lambda i: eng.step_host(h_act[i % 4].numpy(), h_obs.numpy(), h_rew.numpy(), h_done.numpy())
        d2h = (es * (eng.obs_dim + 1) + 1) * n_local
        api = "b747_step_host (C ABI, pinned host buffers; chunked copy/step/copy pipeline replayed as a CUDA graph)"
    for i in range(12):   # warm-up; b747_step_host_packed also settles its host path here (first ten calls)
        step_e2e(i)
    barrier()
    l0 = eng.launch_count
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        step_e2e(i)
    barrier()
    e2e_sec = time.perf_counter() - t0
    te = torch.tensor([e2e_sec], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = n_total * e2e_steps / float(te.item())
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": (4 if dtype == E.F32 else 8) * n_local,
           "d2h_bytes_per_step": d2h, "steps": e2e_steps, "api": api, "gpu_launches": int(eng.launch_count - l0),
           "host_affinity": affinity, "episodes": float(eng.episode_stats()[0])}

    # ---- the only cross-GPU quantity: episode statistics, reduced once
    stats = reduce_episode_stats(stats_timed)
    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = _peaks()
    kernel_ms = sum(per_launch_ms) / len(per_launch_ms)
    extra = {}
    if world == 1 and main_cfg:
        # ---- the same kernel at K = 1 (Controller's default sample_time = dt) and K = 5 (main.py): the K axis
        # (SURVEY.md 8d: only near K = 1 can the step approach the HBM roof)
        def other_k(Kx):
            e1 = E.BatchEngine(n_envs=n_local, dtype=E.F32, device=local_rank, sample_time=Kx * 0.01, seed=1, auto_reset=True)
            e1.use_stream(torch.cuda.current_stream().cuda_stream)
            e1.reset(obs)
            _desync(e1, torch, n_local, int(round(20.0 / (Kx * 0.01))), pool, obs, rew, done, dev)
            for i in range(5):
                e1.step(pool[i % 8], obs, rew, done)
            n1 = max(20, min(args.steps, 200))
            ms1, _ = timed_pass(e1, n1)
            ms1 /= n1
            ach1 = BYTES_PER_ENV_STEP * n_local / (ms1 * 1e-3) / 1e9
            ep1 = float(e1.episode_stats()[0])
            e1.close()
            return {"substeps": Kx, "kernel_ms": ms1, "env_steps_per_s": n_local / (ms1 * 1e-3), "achieved": ach1,
                    "peak": peak, "unit": "GB/s", "frac": ach1 / peak, "steps": n1, "episodes": ep1}
        # secondary measurements never hide the headline: a failure is reported in place of the number
        for key, Kx in (("k1", 1), ("k5", 5)):
            try:
                extra[key] = other_k(Kx)
            except Exception as e:
                extra[key] = {"error": repr(e)}
        # ---- the SB3-facing call: B747VecEnv.step (numpy mode) with float32 [N, 1] actions, terminal observations and
        # monitor records inside the timed region
        try:
            extra_vec = _vecenv_rate(n_local, K, local_rank)
        except Exception as e:
            extra_vec = {"error": repr(e)}
    achieved = bytes_env * n_local / (kernel_ms * 1e-3) / 1e9
    prof = {}
    pj = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if main_cfg and os.path.exists(pj):
        try:
            prof = json.load(open(pj))
        except Exception:
            prof = {}
    kname = {"fp32_1M_K10": "b747::k_env_step32<0, 4, 0, 0>", "tier2_1M_K10": "b747::k_env_step32<2, -1, 0, 0>"}.get(
        args.config, "b747::k_env_step64")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": prof.get("dram_bytes_per_launch"),
                "traffic_source": (f"profiles/ncu_summary.json (ncu --set full capture {prof.get('tag', '?')} of this kernel; not "
                                   "re-measured by this run)") if prof else None,
                "peak_source": peak_src, "bytes_per_env_step": bytes_env, "substeps": K,
                "kernel": kname, "kernel_ms": kernel_ms,
                "note": ("K substeps per launch make the kernel instruction-issue bound, not HBM bound (SURVEY.md 8d); "
                         "pipe utilisation from ncu is in profiles/"),
                "pipes": prof.get("pipes"), "pipes_source": "profiles/ncu_summary.json" if prof else None}
    roofline.update(extra)
    rep_sorted = sorted(rep_ms)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms_total_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": dtype_name, "data": "synthetic",
            "config": _config_dict(args.config),
            "mixed_precision": ("f32 aero/trig/tables, f64 integrator accumulation and pitch-error chain"
                                if dtype == E.F32 else "float64 throughout"),
            "clocks": clocks,
            "repeats": {"n": len(rep_ms), "ms_per_step_min": rep_sorted[0], "ms_per_step_median": rep_sorted[len(rep_sorted) // 2],
                        "ms_per_step_max": rep_sorted[-1],
                        "note": "the timed pass repeated under the clock sampler for >= 0.7 s; `value` is the FIRST pass"},
            "lockstep": {"value": n_total * lock_steps / (lock_ms_max * 1e-3), "unit": UNIT, "ms_per_step": lock_ms_max / lock_steps,
                         "steps": lock_steps, "note": "every env in the same flight phase, no env finishes in the window "
                                                      "(what round 1 reported as `value`)"},
            "e2e": e2e,
            "gpu_launches": int(launches),
            "roofline": roofline,
            "episode_stats": summarize(stats)}
    if world == 1 and main_cfg:
        line["e2e_vecenv"] = extra_vec
    if world == 1 and main_cfg and not args.no_cpu_baseline:
        # BASELINE configs[4]: PPO end to end on a 65536-env GPU VecEnv (torch MLP policy, rollout + update phases replayed as
        # CUDA graphs): env-steps/s including the updates (SB3's time/fps) and wall-clock to the reference's reward level
        try:
            eng.close()
            from b747_rl_ctrl_b200 import ppo
            r = ppo.train(n_envs=65536, threshold=225.0, max_seconds=30.0, seed=1, device=local_rank)
            line["ppo_65536"] = {"steps_per_s": r["steps_per_s"], "seconds": r["seconds"], "steps": r["steps"],
                                 "reached": r["reached"], "final_ep_rew_mean": r["final_ep_rew_mean"], "cuda_graphs": r["graphs"],
                                 "hyper": r["hyper"],
                                 "reference": "ep_rew_mean 225.7 after 98 304 steps at ~340 env-steps/s (4 SubprocVecEnv workers, "
                                              "tensorboard.xlsx; BASELINE.md)"}
        except Exception as e:  # never hides the headline
            line["ppo_65536"] = {"error": repr(e)}
    if world == 1 and not args.no_cpu_baseline:
        try:
            _, info, _ = cpu_reference_rate(3, 1, 300000 if K == 10 else 300000, substeps=K)
            info["python_step_loop"] = python_loop_rate(substeps=K)
            line["cpu_baseline"] = info
        except Exception as e:  # the CPU leg must never hide the GPU number
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "error", "sample": repr(e)}
    if dumped is not None:
        _dump_outputs(args.dump_outputs, dumped, np.float32 if dtype == E.F32 else np.float64)
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


def _vecenv_rate(n, K, device):
    """env-steps/s of B747VecEnv.step_async/step_wait in numpy mode: what stable-baselines3 calls."""
    import numpy as np
    from b747_rl_ctrl_b200.vec_env import B747VecEnv
    out = {"unit": UNIT, "num_envs": n,
           "api": "B747VecEnv.step(actions float32 [N,1]) -> (obs, rew, dones, infos with terminal_observation + episode)"}
    rng = np.random.default_rng(0)
    acts = [rng.uniform(-1, 1, (n, 1)).astype(np.float32) for _ in range(4)]
    for copy in (True, False):
        env = B747VecEnv(n, sample_time=K * 0.01, device=device, copy_outputs=copy)
        env.reset()
        ep_len = int(round(20.0 / (K * 0.01)))
        # spread the episode phases on the device (masked resets while stepping) so that ~1/ep_len of the envs finish --
        # terminal observations, monitor records and info dicts included -- in every timed step
        import torch
        dev = torch.device("cuda", device)
        ids = torch.arange(n, device=dev)
        a_d, o_d, r_d, d_d = env.engine.alloc_io()
        for t in range(ep_len):
            env.engine.step(a_d, o_d, r_d, d_d)
            env.engine.reset(mask=((ids % ep_len) == t).to(torch.uint8))
        env.engine.synchronize()
        del a_d, o_d, r_d, d_d
        for i in range(3):
            env.step(acts[i % 4])
        steps, finished = 10, 0
        t0 = time.perf_counter()
        for i in range(steps):
            _, _, d, infos = env.step(acts[i % 4])
            finished += int(d.sum())
        dt = time.perf_counter() - t0
        out["value" if copy else "value_views"] = n * steps / dt
        out["ms_per_step" if copy else "ms_per_step_views"] = dt / steps * 1e3
        out["episodes_finished"] = finished
        env.close()
    out["note"] = ("value: fresh output arrays every step (SubprocVecEnv semantics); value_views: views of rotating pinned "
                   "buffers (copy_outputs=False).  The step is host-bound: action staging, done unpacking, info dicts.")
    return out


def _dump_outputs(out_dir, arrays, np_dtype):
    """--dump-outputs: every array of the last timed step as <out_dir>/<name>.npy in the handle's float type (done flags
    as 0 / 1), so that two builds can be compared output for output.  The largest configuration writes 20 MiB."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    outs = {name: t.numpy().astype(np_dtype) for name, t in arrays.items()}
    assert sum(a.nbytes for a in outs.values()) <= 64 << 20
    for name, a in outs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _emit(line):
    """The ONE JSON line goes to the real stdout; everything else a library prints (NCCL banner ...) to stderr."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)  # fd 1 -> stderr for the rest of the process (native libraries write to fd 1 directly)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", default="fp32_1M_K10", choices=sorted(CONFIGS),
                    help="fp32_1M_K10 = BASELINE configs[2], the configuration the metric is quoted on (default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write obs, reward and done of the last timed step as DIR/<name>.npy (the envs of GPU 0; the "
                         "inputs are seeded, so equal arguments give equal inputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs applies to --impl cuda")
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # convenience launcher: re-exec under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(29400 + os.getpid() % 500), os.path.abspath(__file__),
               "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup), "--config", args.config]
        if args.dump_outputs:
            cmd += ["--dump-outputs", args.dump_outputs]
        sys.exit(subprocess.call(cmd))
    run_cuda(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
