"""Copy rates of b747_save_state / b747_load_state against a plain device-to-device cudaMemcpyAsync of the same bytes.

  * save all / load all of 1 Mi canonical f32 envs (identity index maps: one blob row per state row);
  * a 1 Ki-env blob broadcast-loaded into 1 Mi envs (blob_idx = k % 1024, the fan-out of a search baseline);
  * torch's same-dtype device copy of a uint8 tensor of the blob's size (one cudaMemcpyAsync) as the reference.

Call times come from CUDA events on the stream doing the work, over `reps` back-to-back calls after warm-up (a load
also reads the blob header back and synchronises, so its call time holds one host round trip); kernel times come from
torch.profiler in a separate pass.  The working set (2 x 331 MB) is larger than the 126 MB L2.  Rates are copy bytes
per second: blob payload bytes (without the 64-byte header) over time; each byte is read once and written once.  The
card's name and power limit are read in the same run.  Usage: python tools/state_probe.py [n_envs] [reps] [--out file.json]
"""
import ctypes
import json
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from b747_rl_ctrl_b200 import engine as E  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
if out_path in args:
    args.remove(out_path)
n = int(args[0]) if args else 1 << 20
reps = int(args[1]) if len(args) > 1 else 20
dev = torch.device("cuda", 0)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in q.split(",")]
        return name, power
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def timed(fn, stream):
    """ms per call: CUDA events on `stream` around `reps` calls (after 3 warm-up calls)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(reps):
        fn()
    b.record(stream)
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def kernel_ms(fn, calls=5):
    """Mean device time of the kernels / copies one call issues (torch.profiler, CUDA activity), in a profiled
    pass of its own after the timed one."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    busy = [e for e in prof.events() if str(e.device_type).endswith("CUDA") and
            ("k_state_copy" in e.name or "DtoD" in e.name or "Device -> Device" in e.name)]
    return sum(e.time_range.elapsed_us() for e in busy) / 1e3 / calls if busy else None


eng = E.BatchEngine(n_envs=n, dtype=E.F32, sample_time=0.1, seed=1)
eng.reset()
h_stream = torch.cuda.ExternalStream(eng.stream_ptr, device=dev)
nb = eng.state_bytes()
payload = nb - 64
blob = torch.empty(nb, dtype=torch.uint8, device=dev)
eng.save_state(out=blob)
res = dict(n_envs=n, reps=reps, blob_bytes=nb, bytes_per_env=payload / n)

raw = eng._L


def ok(rc):
    assert rc == 0, raw.b747_last_error()


vp = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
small = E.BatchEngine(n_envs=1024, dtype=E.F32, sample_time=0.1, seed=2)
small.reset()
sblob = small.save_state()
bidx = (torch.arange(n, dtype=torch.int32, device=dev) % 1024).contiguous()
src = torch.empty(payload, dtype=torch.uint8, device=dev).random_(0, 255)
dst = torch.empty_like(src)
torch.cuda.synchronize()
cur = torch.cuda.current_stream(dev)
# the C ABI directly (no Python-side checks): save is asynchronous, load reads the 64-byte header back and synchronises
cases = {
    "save_all": (lambda: ok(raw.b747_save_state(eng._h, None, n, vp(blob))), h_stream),
    "load_all": (lambda: ok(raw.b747_load_state(eng._h, vp(blob), None, None, n)), h_stream),
    "broadcast_1Ki_to_all": (lambda: ok(raw.b747_load_state(eng._h, vp(sblob), vp(bidx), None, n)), h_stream),
    "memcpy_d2d": (lambda: dst.copy_(src), cur),
}
for name, (fn, stream) in cases.items():
    ms = timed(fn, stream)
    res[name] = dict(call_ms=ms, call_GBps=payload / ms / 1e6)
    kern = kernel_ms(fn)
    if kern:
        res[name].update(kernel_ms=kern, kernel_GBps=payload / kern / 1e6)
for k in ("save_all", "load_all", "broadcast_1Ki_to_all"):
    for t in ("call", "kernel"):
        if f"{t}_GBps" in res[k] and f"{t}_GBps" in res["memcpy_d2d"]:
            res[k][f"{t}_of_memcpy"] = res[k][f"{t}_GBps"] / res["memcpy_d2d"][f"{t}_GBps"]

# the copies are exact: a reloaded blob saves back to the same bytes
eng.load_state(blob)
again = eng.save_state()
torch.cuda.synchronize()
res["round_trip_exact"] = bool(torch.equal(again, blob))
res["card"], res["power_limit"] = card()
line = json.dumps(res)
print(line)
if out_path:
    with open(out_path, "w") as f:
        f.write(line + "\n")
eng.close()
small.close()
