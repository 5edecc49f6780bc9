"""The f32 step kernels in the multi-tile regime they run in at scale.

Every f32 step kernel is persistent: grid = SMs x resident blocks, each warp steps a fixed first tile of 32 envs and then
takes further tiles from a per-launch counter (or, in the TMA-staged K = 1 kernel, walks a static stride with the next
tile's state already in flight).  With N = 2^18 + 77 envs every warp steps three or more tiles and the last tile is
ragged.  For every reachable instantiation (TIER, SW, STG, PFA) this module
  * profiles one launch and checks that the intended kernel ran with fewer resident threads than envs;
  * steps the same seeded actions through that kernel (more than 64 launches back to back, so the 64-slot tile-counter
    ring wraps) and through a second handle whose step_host pipeline cuts every launch down to at most one tile per warp
    (set_host_chunks(64)), and asserts that both give the same bits: outputs at every step, every per-env field at the
    end, signals / transfer metrics / recorder on the full tier;
  * replays the episode bookkeeping on the host (ep_return += (double)rew in step order) against last_episode() and
    episode_stats();
  * compares three 256-env slices with the float64 oracle -- the first envs, the first tiles the counter hands out and
    the ragged tail -- under test_gpu_parity's per-family bounds and flight-envelope excusal.
"""
import json
import math
import os
import re
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
from test_gpu_parity import FAMILY_BOUNDS, REW_JUMP, _envelope_update, _reward_edge  # noqa: E402

pytestmark = pytest.mark.gpu

N = (1 << 18) + 77
STEPS = 72          # the first step is profiled, the other 71 are launched with no host synchronisation in between
SINGLE_TILE_CHUNKS = 64    # single-tile form: 63 chunk launches of <= 4224 envs = 132 tiles, fewer than any tier's resident warps
SW_RP = 4           # MP32 switch word with use_RP alone (b747_model_mx.cuh): the canonical compile-time setting
K1 = dict(sample_time=0.01, tk=0.3)   # 30-step episodes
K5 = dict(sample_time=0.05, tk=1.0)   # 20-step episodes

# Bounds of the two runtime-switch families (|d obs| / (1 + |obs|), |d reward|, share of env-steps outside the envelope):
# measured maxima over the three slices of this module with a margin of about 3x (B200: use_RP = 0 on the canonical
# family 3.0e-8 / 1.4e-6, use_RL = 1 on the ADD_PROC speed family 3.0e-7 / 4.0e-6; no env left the envelope).
SWITCH_BOUNDS = {
    "T0-SW": (1e-7, 5e-6, 0.02),
    "T1-SW": (1e-6, 1.2e-5, 0.02),
}

# config -> engine / oracle keywords, engine-only keywords, set_param applied to the handles and every oracle env,
# the entry points stepped in the multi-tile form with the kernel each must launch (TIER, SW, STG, PFA), bounds
CASES = {
    "T0-K1": dict(kw=K1, forms={"step": (0, SW_RP, 1, 0), "packed": (0, SW_RP, 1, 0), "host_packed": (0, SW_RP, 0, 1)},
                  bounds=FAMILY_BOUNDS["K1_tk3"]),
    "T0": dict(kw=K5, forms={"step": (0, SW_RP, 0, 0)}, bounds=FAMILY_BOUNDS["K10"]),
    "T0-SW": dict(kw=K5, param=("use_RP", 0.0), forms={"step": (0, -1, 0, 0)}, bounds=SWITCH_BOUNDS["T0-SW"]),
    "T1": dict(kw=dict(obs_type=1, ctrl_mode=1, action_max=1.0, **K5), forms={"step": (1, SW_RP, 0, 0)},
               bounds=FAMILY_BOUNDS["speed_addproc"]),
    "T1-SW": dict(kw=dict(obs_type=1, ctrl_mode=1, action_max=1.0, **K5), param=("use_RL", 1.0),
                  forms={"step": (1, -1, 0, 0)}, bounds=SWITCH_BOUNDS["T1-SW"]),
    "T2": dict(kw=dict(rew_type=2, ctrl_type=2, reset_ref_mode=2, **K5), forms={"step": (2, -1, 0, 0)},
               bounds=FAMILY_BOUNDS["quality_semimanual"]),
    "T3": dict(kw=K5, ekw=dict(export_signals=True, track_transfer=True, record_capacity=12),
               forms={"step": (3, -1, 0, 0)}, bounds=FAMILY_BOUNDS["K10"]),
}
BOOK_FIELDS = ("tick", "flags", "ep_idx", "last_ret", "last_len")


def _bits(x):
    return np.ascontiguousarray(x).view(np.uint8)


def _diff(what, x, y):
    """'' if x and y hold the same bits, else where they first differ."""
    if x.shape == y.shape and np.array_equal(_bits(x), _bits(y)):
        return ""
    if x.shape != y.shape:
        return f"{what}: shapes {x.shape} / {y.shape}"
    d = _bits(x).reshape(len(x), -1) != _bits(y).reshape(len(y), -1)
    envs = np.nonzero(d.any(axis=1))[0]
    return f"{what}: {len(envs)} envs differ, first {envs[:5].tolist()} ({x[envs[0]]} / {y[envs[0]]})"


def _template_args(name):
    """(TIER, SW, STG, PFA) from a demangled k_env_step32<...> name, bools printed as true/false or as integers."""
    m = re.search(r"k_env_step32<([^>]*)>", name)
    assert m, name
    args = [re.sub(r"\(\w+\)", "", a).strip() for a in m.group(1).split(",")]
    return tuple({"true": 1, "false": 0}[a] if a in ("true", "false") else int(a) for a in args)


def _profiled(fn, path):
    """k_env_step32 launches of fn() as chrome-trace kernel events of torch.profiler (CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    return [e for e in events if e.get("cat") == "kernel" and "k_env_step32" in e.get("name", "")]


def _episode_book(rew, done):
    """Host replay of the kernel's bookkeeping: each env's float32 rewards summed into float64 in step order."""
    ret = np.zeros(N)
    ln = np.zeros(N, np.int64)
    last_ret, last_len = np.zeros(N), np.zeros(N, np.int64)
    stats = np.zeros(4)
    rets = []
    for k in range(len(rew)):
        ret += rew[k].astype(np.float64)
        ln += 1
        d = done[k].astype(bool)
        last_ret[d], last_len[d] = ret[d], ln[d]
        rets.append(ret[d].copy())
        stats[0] += d.sum()
        stats[2] += ln[d].sum()
        ret[d], ln[d] = 0.0, 0
    r = np.concatenate(rets)
    stats[1], stats[3] = math.fsum(r), math.fsum(r * r)
    return last_ret, last_len, stats


class Run:
    """Outcome of one configuration: the kernels that ran, every bit-level difference between the multi-tile forms and
    the single-tile form, the bookkeeping read back from each handle, the oracle deviations per slice."""


def _make(E, name, n_chunks=None):
    c = CASES[name]
    eng = E.BatchEngine(n_envs=N, dtype=E.F32, seed=17, auto_reset=True, **c["kw"], **c.get("ekw", {}))
    if "param" in c:
        eng.set_param(c["param"][0], [c["param"][1]])
    if n_chunks:
        eng.set_host_chunks(n_chunks)
    eng.reset()
    return eng


def _step_forms(E, name, acts, tmp):
    """Multi-tile forms: {form: (handle, kernel events of the profiled first step, host history)}."""
    import torch
    dev = torch.device("cuda")
    c = CASES[name]
    acts_d = torch.from_numpy(acts).to(dev)
    torch.cuda.synchronize()
    out = {}
    for form in c["forms"]:
        eng = _make(E, name)
        od, rf, nw = eng.obs_dim, eng.record_floats, (N + 31) // 32
        if form == "step":
            obs = torch.empty(STEPS, N, od, device=dev)
            rew = torch.empty(STEPS, N, device=dev)
            done = torch.empty(STEPS, N, dtype=torch.uint8, device=dev)
            term = torch.empty(STEPS, N, od, device=dev)

            def one(k):
                eng.step(acts_d[k], obs[k], rew[k], done[k], term[k])
        elif form == "packed":
            rec = torch.empty(STEPS, N, rf, device=dev)
            bits = torch.empty(STEPS, nw, dtype=torch.int32, device=dev)

            def one(k):
                eng.step_packed(acts_d[k], rec[k], bits[k])
        else:   # zero-copy both ways: the kernel reads the next tile's actions from pinned host memory
            eng.set_host_mode(2)
            a_p = torch.empty(N).pin_memory()
            r_p = torch.empty(N, rf).pin_memory()
            b_p = torch.empty(nw, dtype=torch.int32).pin_memory()
            rec_h = np.empty((STEPS, N, rf), np.float32)
            bits_h = np.empty((STEPS, nw), np.int32)

            def one(k):
                a_p.numpy()[:] = acts[k]
                eng.step_host_packed(a_p.numpy(), r_p.numpy(), b_p.numpy())
                rec_h[k], bits_h[k] = r_p.numpy(), b_p.numpy()

        ev = _profiled(lambda: (one(0), eng.synchronize()), tmp / f"{name}_{form}.pt.trace.json")
        for k in range(1, STEPS):
            one(k)
        eng.synchronize()
        if form == "step":
            h = dict(obs=obs.cpu().numpy(), rew=rew.cpu().numpy(), done=done.cpu().numpy(), term=term.cpu().numpy())
            del obs, rew, done, term
        else:
            if form == "packed":
                rec_h, bits_h = rec.cpu().numpy(), bits.cpu().numpy()
                del rec, bits
            d = np.unpackbits(bits_h.view(np.uint8).reshape(STEPS, -1), axis=1, bitorder="little")[:, :N]
            h = dict(rew=rec_h[:, :, od], done=d, term=rec_h[:, :, :od], pad=rec_h[:, :, od + 1:])
        out[form] = (eng, ev, h)
    del acts_d
    return out


def _fields(eng):
    from b747_rl_ctrl_b200 import engine as E
    got = {}
    for f in eng.field_names():
        try:
            got[f] = eng.get(f)
        except E.B747Error:
            got[f] = None   # not carried by an f32 handle
    return got


def _oracle_slices(O, name, acts, hist, resident):
    """Worst deviations of three 256-env slices of the multi-tile run from the float64 oracle."""
    c = CASES[name]
    cfg_o = O.make_cfg(seed=17, **c["kw"])
    res = {}
    for tag, lo in (("first", 0), ("counter", resident), ("tail", N - 256)):
        m = 256
        ob = O.OracleBatch(cfg_o, m, env_id_offset=lo)
        ob.reset()
        if "param" in c:
            for i in range(m):
                ob.model(i).set(*c["param"])
        out = np.zeros(m, bool)
        r = dict(lo=lo, obs=0.0, rew=0.0, rew_edge=0.0, excused=0, total=0, done_diff=[], n_done=0)
        for k in range(STEPS):
            o_o, r_o, d_o, t_o = ob.step(acts[k, lo:lo + m].astype(np.float64))
            if not np.array_equal(hist["done"][k, lo:lo + m].astype(bool), d_o):
                r["done_diff"].append(k)
            r["n_done"] += int(d_o.sum())
            inside = _envelope_update(ob, out, d_o)
            eo = (np.abs(hist["term"][k, lo:lo + m].astype(np.float64) - t_o) / (1.0 + np.abs(t_o))).max(axis=1)
            er = np.abs(hist["rew"][k, lo:lo + m].astype(np.float64) - r_o)
            edge = _reward_edge(O, cfg_o, ob, t_o, d_o)
            r["obs"] = max(r["obs"], float(eo[inside].max(initial=0.0)))
            r["rew"] = max(r["rew"], float(er[inside & ~edge].max(initial=0.0)))
            r["rew_edge"] = max(r["rew_edge"], float(er[inside & edge].max(initial=0.0)))
            r["excused"] += int(out.sum())
            r["total"] += m
            out &= ~d_o
        res[tag] = r
    return res


@pytest.fixture(scope="module", params=sorted(CASES))
def run(request, oracle, tmp_path_factory):
    import torch
    assert torch.cuda.is_available()
    from b747_rl_ctrl_b200 import engine as E
    name = request.param
    c = CASES[name]
    acts = np.random.default_rng(29).uniform(-1.0, 1.0, (STEPS, N)).astype(np.float32)
    R = Run()
    R.name = name
    forms = _step_forms(E, name, acts, tmp_path_factory.mktemp(name))
    R.kernels = {f: ev for f, (_, ev, _) in forms.items()}
    # single-tile form: every chunk launch gives each warp at most one tile
    ref = _make(E, name, n_chunks=SINGLE_TILE_CHUNKS)
    od = ref.obs_dim
    R.diffs = []
    hist_b = dict(obs=[], rew=[], done=[], term=[])
    for k in range(STEPS):
        cur = dict(zip(("obs", "rew", "done", "term"), ref.step_host(acts[k], terminal_obs=np.empty((N, od), np.float32))))
        for key, v in cur.items():
            hist_b[key].append(v)
        for f, (_, _, h) in forms.items():
            for key, v in cur.items():
                if key in h:   # packed records carry no post-reset observation
                    d = _diff(f"{f} step {k} {key}", h[key][k], v)
                    if d:
                        R.diffs.append(d)
            if "pad" in h and (h["pad"][k] != 0).any():
                R.diffs.append(f"{f} step {k}: non-zero record padding")
    # every per-env field an f32 handle returns, after the last step
    fb = _fields(ref)
    R.fields = sorted(k for k, v in fb.items() if v is not None)
    for f, (eng, _, _) in forms.items():
        fa = _fields(eng)
        for k in fb:
            if (fa[k] is None) != (fb[k] is None):
                R.diffs.append(f"{f} field {k}: available on one handle only")
            elif fb[k] is not None:
                d = _diff(f"{f} field {k}", fa[k], fb[k])
                if d:
                    R.diffs.append(d)
    first = next(iter(forms))
    ev = R.kernels[first]
    resident = ev[0]["args"]["grid"][0] * ev[0]["args"]["block"][0] if ev else 0   # threads = 32 x resident warps
    if "ekw" in c:   # full tier: transfer metrics and recorder
        eng = forms["step"][0]
        for which in ("SS", "CS"):
            for fin in (True, False):
                d = _diff(f"transfer_metrics {which} finished={fin}", eng.transfer_metrics(which, fin),
                          ref.transfer_metrics(which, fin))
                if d:
                    R.diffs.append(d)
        R.recorded = [resident + 5, 2 * resident + 77, N - 13, N - 1]
        for i in R.recorded:
            ra, rb = eng.recorder_read(i), ref.recorder_read(i)
            assert len(rb["t"]) == c["ekw"]["record_capacity"]
            for key in rb:
                d = _diff(f"recorder env {i} {key}", ra[key], rb[key])
                if d:
                    R.diffs.append(d)
    # bookkeeping: replayed from the single-tile outputs (the comparison above ties the other forms to them)
    rew_b, done_b = np.stack(hist_b["rew"]), np.stack(hist_b["done"])
    R.book_expected = _episode_book(rew_b, done_b)
    R.book = {f: (eng.last_episode(), eng.episode_stats()) for f, (eng, _, _) in forms.items()}
    R.book["single-tile"] = (ref.last_episode(), ref.episode_stats())
    # oracle on slices of the (first) multi-tile form
    R.resident = resident
    hist = forms[first][2]
    R.oracle = _oracle_slices(oracle, name, acts, hist, resident) if resident else {}
    for f, (eng, _, _) in forms.items():
        eng.close()
    ref.close()
    del forms, hist, hist_b
    torch.cuda.empty_cache()
    return R


def test_intended_kernel_runs_multi_tile(run):
    """Each entry point launches the instantiation the table names, with fewer resident threads than envs."""
    for form, want in CASES[run.name]["forms"].items():
        ev = run.kernels[form]
        assert len(ev) == 1, f"{run.name}/{form}: expected one k_env_step32 launch in the profiled step, got {len(ev)}"
        e = ev[0]
        grid, block = e["args"]["grid"], e["args"]["block"]
        threads = grid[0] * block[0]
        print(f"{run.name}/{form}: {e['name'].split('(')[0]} grid {grid} block {block}, "
              f"{(N + 31) // 32 / (threads // 32):.2f} tiles per warp")
        assert _template_args(e["name"]) == want, e["name"]
        assert threads < N, f"{run.name}/{form}: {threads} resident threads cover all {N} envs"


def test_multi_tile_equals_single_tile_bit_for_bit(run):
    """Outputs at every step, every per-env field, signals / transfer metrics / recorder: same bits whether the warps
    walk several tiles per launch or one."""
    assert set(BOOK_FIELDS) <= set(run.fields)
    if "ekw" in CASES[run.name]:
        assert sum(f.startswith("sig_") for f in run.fields) >= 30
    assert not run.diffs, f"{len(run.diffs)} differences, first: " + "; ".join(run.diffs[:5])


def test_episode_bookkeeping_exact(run):
    """last_episode() reproduces the host's float64 sum of each env's rewards bit for bit; episode_stats() counts and
    lengths exactly, sums of returns and of squared returns up to the order of the float64 atomics."""
    last_ret, last_len, st = run.book_expected
    assert st[0] >= N   # every env finished at least one episode inside the run
    for form, ((ret, ln), got) in run.book.items():
        assert np.array_equal(ret.view(np.uint64), last_ret.view(np.uint64)), form
        assert np.array_equal(ln, last_len), form
        assert got[0] == st[0] and got[2] == st[2], (form, got, st)
        assert abs(got[1] - st[1]) <= 1e-12 * abs(st[1]), (form, got[1], st[1])
        assert abs(got[3] - st[3]) <= 1e-12 * abs(st[3]), (form, got[3], st[3])


def test_counter_scheduled_tiles_match_oracle(run):
    """The first envs, the first tiles the counter (or the static stride) hands out and the ragged tail, against the
    float64 oracle: done flags bit-exact, observation and reward within the family's bound inside the envelope."""
    ob_bound, rew_bound, max_ex = CASES[run.name]["bounds"]
    assert run.resident and run.oracle
    for tag, r in run.oracle.items():
        print(f"{run.name} oracle slice {tag} (envs {r['lo']}..{r['lo'] + 255}): |d obs|/(1+|obs|) {r['obs']:.2e} "
              f"(bound {ob_bound:.0e}), |d rew| {r['rew']:.2e} (bound {rew_bound:.0e}), at a reward edge "
              f"{r['rew_edge']:.2e}; excused {r['excused']} of {r['total']} env-steps; episodes {r['n_done']}")
    for tag, r in run.oracle.items():
        assert not r["done_diff"], f"{tag}: done flags differ at steps {r['done_diff'][:5]}"
        assert r["n_done"] >= 256
        assert r["obs"] <= ob_bound, (tag, r)
        assert r["rew"] <= rew_bound, (tag, r)
        assert r["rew_edge"] <= rew_bound + REW_JUMP, (tag, r)
        assert r["excused"] <= max_ex * r["total"], (tag, r)
