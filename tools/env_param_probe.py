"""Step time of the per-env twins (b747_set_env_param) against the whole-batch kernels they shadow.

Rows, each a pair of handles stepped alternately in one process (K = 10, tk = 20 s: 200-step episodes, phases spread
as bench.py does, so ~1/200 of the envs auto-reset in every launch):
  * tier 0 (canonical, whole-batch)  vs  the tier-1 twin with fixed per-env values  vs  the tier-1 twin with ranges on
    every name (redraws at each auto-reset) -- 1 Mi envs;
  * tier 2 (HYBRID reset) vs its twin -- 1 Mi envs;
  * float64 vs its twin -- 256 Ki envs.
Per-env values equal the batch values, so every handle flies the same episodes.  Times are CUDA events on the handle's
stream around `reps` back-to-back device steps, repeated `rounds` times with the handles alternating; the median round
is reported.  The working sets are larger than the 126 MB L2.  The card's name and power limit are read in the same run.
Usage: python tools/env_param_probe.py [reps] [rounds] [--out file.json]
"""
import json
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
from b747_rl_ctrl_b200 import engine as E  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
if out_path in args:
    args.remove(out_path)
reps = int(args[0]) if args else 20
rounds = int(args[1]) if len(args) > 1 else 5
dev = torch.device("cuda", 0)
K, TK, EP_LEN = 10, 20.0, 200
RANGES = {"m0": (2.6e5, 3.4e5), "Iz": (3.5e7, 4.5e7), "P": (3.4e5, 3.8e5), "S": (500.0, 530.0), "c_": (8.0, 8.6),
          "PID_SS": ([-2.5, 0.2, -0.7, 20], [-1.5, 0.4, -0.3, 30]), "PID_CS": ([0.002, 2e-5, 0.02, 8], [0.006, 6e-5, 0.06, 12])}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in q.split(",")]
        return name, power
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def make(n, dtype, mode, **kw):
    eng = E.BatchEngine(n_envs=n, dtype=dtype, sample_time=K * 0.01, tk=TK, seed=1, **kw)
    if mode == "fixed":
        eng.set_env_param("m0", np.full(n, eng.get_param("m0")))
    elif mode == "ranges":
        for nm, (lo, hi) in RANGES.items():
            eng.set_env_param_range(nm, lo, hi)
    tdt = torch.float32 if dtype == E.F32 else torch.float64
    bufs = eng.alloc_io()
    g = torch.Generator(device=dev).manual_seed(3)
    pool = [torch.rand(n, device=dev, generator=g, dtype=tdt) * 2 - 1 for _ in range(4)]
    eng.reset()
    ids = torch.arange(n, device=dev)
    for t in range(EP_LEN):  # bench.py's phase spread: a masked reset of the envs id % EP_LEN == t at step t
        eng.step(pool[t % 4], *bufs[1:])
        eng.reset(mask=((ids % EP_LEN) == t).to(torch.uint8))
    eng.synchronize()
    return eng, bufs, pool


def time_steps(eng, bufs, pool):
    s = torch.cuda.ExternalStream(eng.stream_ptr, device=dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(s)
    for k in range(reps):
        eng.step(pool[k % 4], *bufs[1:])
    b.record(s)
    b.synchronize()
    return a.elapsed_time(b) / reps


def compare(label, specs):
    hs = {name: make(*spec[:3], **spec[3]) for name, spec in specs.items()}
    for name, h in hs.items():  # warm-up of the timed shapes
        time_steps(*h)
    t = {name: [] for name in hs}
    for _ in range(rounds):
        for name, h in hs.items():
            t[name].append(time_steps(*h))
    res = {}
    for name, ts in t.items():
        n = specs[name][0]
        ms = float(np.median(ts))
        res[name] = {"n_envs": n, "ms_per_step": ms, "env_steps_per_s": n / (ms * 1e-3),
                     "spread_ms": [float(min(ts)), float(max(ts))]}
    base = next(iter(res))
    for name in res:
        res[name]["vs_" + base] = res[name]["ms_per_step"] / res[base]["ms_per_step"]
        print(f"{label:10s} {name:22s} {res[name]['ms_per_step']:.4f} ms/step ({res[name]['env_steps_per_s']:.3e} "
              f"env-steps/s, x{res[name]['vs_' + base]:.3f}; rounds {res[name]['spread_ms'][0]:.4f}-"
              f"{res[name]['spread_ms'][1]:.4f})", flush=True)
    for h in hs.values():
        h[0].close()
    return res


name, power = card()
print(f"card: {name}, power limit {power}; K = {K}, {reps} steps x {rounds} rounds per handle", flush=True)
N = 1 << 20
report = {"card": name, "power_limit": power, "K": K, "reps": reps, "rounds": rounds}
report["tier1"] = compare("tier 0/1", {"tier0": (N, E.F32, "batch", {}), "tier1_twin_fixed": (N, E.F32, "fixed", {}),
                                       "tier1_twin_ranges": (N, E.F32, "ranges", {})})
report["tier2"] = compare("tier 2", {"tier2": (N, E.F32, "batch", dict(reset_ref_mode=2)),
                                     "tier2_twin": (N, E.F32, "fixed", dict(reset_ref_mode=2))})
report["f64"] = compare("f64", {"f64": (1 << 18, E.F64, "batch", {}), "f64_twin": (1 << 18, E.F64, "fixed", {})})
if out_path:
    with open(out_path, "w") as f:
        json.dump(report, f, indent=1)
