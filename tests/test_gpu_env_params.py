"""Per-env airframe parameters and PID gains (b747_set_env_param / b747_get_env_param / b747_set_env_param_range,
BatchEngine.set_env_param ..., B747VecEnv(param_ranges=...)).

  * per-env equals whole-batch: one per-env handle whose env groups carry different parameter sets steps bit for bit
    like one whole-batch handle per group (same env ids through env_id_offset), across auto-resets, for the f32 tier 1,
    2 and 3 twins (one of them at 2^18 + 77 envs), float64 with signals and float64 raw model stepping;
  * routing: the twins run by template arguments, a canonical handle without per-env mode still runs tier 0;
  * draws: ranged values equal lo + (hi - lo) u with u recomputed from b747_philox4x32 at the documented counter, the
    episode draws do not move, masked resets redraw masked envs only, explicit episodes and loads leave values alone;
  * against the float64 oracle with every per-env component drawn at every reset, the oracle computing the draws
    itself; tunables survive HYBRID resets (unlike the reference's re-created Model);
  * the API's argument checks, index conventions, set_param broadcasting, the fork recipe and the VecEnv option.
"""
import ctypes
import math
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)

from test_gpu_parity import ROW0, TUNED_SCALE  # noqa: E402

pytestmark = pytest.mark.gpu

N_BIG = (1 << 18) + 77
K5 = dict(sample_time=0.05, tk=1.0)  # 20-step episodes
NAMES = ("m0", "Iz", "P", "S", "c_", "PID_SS", "PID_CS")
# multipliers of the whole-batch defaults for the second parameter set (the first set is the defaults themselves)
SCALE = {nm: TUNED_SCALE[nm] for nm in NAMES}


def _bits(x):
    x = x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)
    return np.ascontiguousarray(x).view(np.uint8)


def _same(a, b):
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
    b = b.cpu().numpy() if hasattr(b, "cpu") else np.asarray(b)
    return a.shape == b.shape and np.array_equal(_bits(a), _bits(b))


@pytest.fixture(scope="module")
def E():
    import torch
    assert torch.cuda.is_available()
    from b747_rl_ctrl_b200 import engine
    return engine


def _param_set(eng, g):
    """Parameter set of group g: the handle's whole-batch values (g = 0) or them scaled by SCALE."""
    out = {}
    for nm in NAMES:
        v = np.atleast_1d(eng.get_param(nm, E_N(nm)))
        out[nm] = v if g == 0 else v * np.asarray(SCALE[nm])
    return out


def E_N(nm):
    return 4 if nm.startswith("PID") else 1


def _fields(eng):
    out = {}
    for nm in eng.field_names():
        try:
            out[nm] = eng.get(nm)
        except Exception:
            pass
    return out


def _concat(parts):
    return np.concatenate(parts, axis=0)


def _evaluation(eng, envs):
    """last_episode, transfer metrics and recorder rows of envs (where the handle has them)."""
    out = {"last": eng.last_episode()}
    if eng.cfg.track_transfer:
        out["tm"] = (eng.transfer_metrics("SS", False), eng.transfer_metrics("CS", True))
    if eng.cfg.record_capacity:
        out["rec"] = [eng.recorder_read(int(i)) for i in envs]
    return out


CASES = {  # obs_bound: DESIGN.md 4.2 family bound of the configuration (SPEED obs / ADD_PROC, QUALITY / SEMI / HYBRID,
           # canonical)
    "f32-T1": dict(f32=True, kw=dict(obs_type=1, ctrl_mode=1, action_max=1.0, **K5), packed=True, n=N_BIG, obs_bound=3e-4),
    "f32-T2": dict(f32=True, kw=dict(rew_type=2, ctrl_type=2, reset_ref_mode=2, **K5), n=3000, obs_bound=5e-4),
    "f32-T3": dict(f32=True, kw=dict(export_signals=True, track_transfer=True, record_capacity=16, **K5), n=3000,
                   obs_bound=1e-6),
    "f64": dict(f32=False, kw=dict(export_signals=True, track_transfer=True, record_capacity=16, **K5), n=1000),
}


@pytest.mark.parametrize("case", list(CASES))
def test_per_env_equals_whole_batch(E, case):
    """Group g of the per-env handle (envs [start_g, start_g + n_g)) against a handle of n_g envs at env_id_offset
    start_g that flies p_g for every env: outputs, every field, signals, last_episode, episode statistics, transfer
    metrics and recorder rows identical at every step, over 50 steps (two and a half episodes).
    float64: the reference is a whole-batch handle with set_param(p_g) -- same bits (-fmad=false, same expressions).
    f32: the reference is a per-env handle holding p_g in every env (the same twin).  Against whole-batch f32 handles the
    twin is not bit-identical: nvcc may contract a product and a sum into one FMA differently in the twin and in the plain
    tier (e.g. the altitude-loop `e_h * PID_CS[0] + csi + cs_d`), and the plain tiers' code is left as it is.  Such
    last-bit differences grow without bound in a chaotic trajectory, so the whole-batch handles are reloaded with the
    per-env handle's state (b747_load_state; parameters stay out of the blob) before each compared step: one env step
    from the same state must give the same done flags and observations within the configuration family's bound of
    DESIGN.md 4.2 (d obs / (1 + |obs|))."""
    cs = CASES[case]
    dt = E.F32 if cs["f32"] else E.F64
    n = cs["n"]
    sizes = [n // 2, n - n // 2]
    starts = [0, sizes[0]]
    per = E.BatchEngine(n_envs=n, dtype=dt, seed=11, **cs["kw"])
    whole_b = [E.BatchEngine(n_envs=sizes[g], dtype=dt, seed=11, env_id_offset=starts[g], **cs["kw"]) for g in range(2)]
    psets = [_param_set(per, g) for g in range(2)]
    for g in range(2):
        for nm, v in psets[g].items():
            whole_b[g].set_param(nm, v)
    if cs["f32"]:
        whole = [E.BatchEngine(n_envs=sizes[g], dtype=dt, seed=11, env_id_offset=starts[g], **cs["kw"]) for g in range(2)]
        for g in range(2):
            for nm, v in psets[g].items():
                whole[g].set_env_param(nm, np.tile(v, (sizes[g], 1)) if E_N(nm) > 1 else np.full(sizes[g], v[0]))
    else:
        whole = whole_b
    for nm in NAMES:
        vals = _concat([np.tile(psets[g][nm], (sizes[g], 1)) for g in range(2)])
        per.set_env_param(nm, vals if E_N(nm) > 1 else vals[:, 0])
    for eng in {id(e): e for e in [per] + whole + whole_b}.values():
        eng.reset()
    d_batch = 0.0
    rng = np.random.default_rng(5)
    packed = cs.get("packed", False)
    rf = per.record_floats if packed and cs["f32"] else 0
    for k in range(50):
        a = rng.uniform(-1, 1, n).astype(per.np_dtype)
        if packed and k % 2:
            out = np.zeros((n, rf), np.float32)
            bits = np.zeros((n + 31) // 32, np.uint32)
            per.step_host_packed(a, out, bits)
            wo = []
            for g in range(2):
                o = np.zeros((sizes[g], rf), np.float32)
                b = np.zeros((sizes[g] + 31) // 32, np.uint32)
                whole[g].step_host_packed(a[starts[g]:starts[g] + sizes[g]], o, b)
                wo.append(o)
            assert _same(out, _concat(wo)), f"{case}: packed records differ at step {k}"
        else:
            if whole_b is not whole:  # the whole-batch handles start this step from the per-env handle's state
                blob = per.save_state()
                for g in range(2):
                    whole_b[g].load_state(blob, blob_indices=np.arange(starts[g], starts[g] + sizes[g], dtype=np.int32))
            obs, rew, done = per.step_host(a)
            res = [whole[g].step_host(a[starts[g]:starts[g] + sizes[g]]) for g in range(2)]
            assert _same(obs, _concat([r[0] for r in res])), f"{case}: obs differ at step {k}"
            assert _same(rew, _concat([r[1] for r in res])), f"{case}: rewards differ at step {k}"
            assert _same(done, _concat([r[2] for r in res])), f"{case}: done flags differ at step {k}"
            if whole_b is not whole:
                rb = [whole_b[g].step_host(a[starts[g]:starts[g] + sizes[g]]) for g in range(2)]
                ob = _concat([r[0] for r in rb])
                assert _same(done, _concat([r[2] for r in rb])), f"{case}: done flags differ from whole-batch at {k}"
                d_batch = max(d_batch, float((np.abs(obs - ob) / (1 + np.abs(ob))).max()))
                assert d_batch <= cs["obs_bound"], f"{case}: twin and whole-batch tier apart by {d_batch:.3e} at step {k}"
        if k % 10 == 9 or k == 49:
            fp = _fields(per)
            fw = [_fields(w) for w in whole]
            assert set(fp) == set(fw[0])
            for nm in fp:
                assert _same(fp[nm], _concat([f[nm] for f in fw])), f"{case}: field {nm} differs at step {k}"
            ep = _evaluation(per, [0, starts[1]])
            ew = [_evaluation(whole[g], [0]) for g in range(2)]
            for j in range(2):
                assert _same(ep["last"][j], _concat([e["last"][j] for e in ew]))
            if "tm" in ep:
                for j in range(2):
                    assert _same(ep["tm"][j], _concat([e["tm"][j] for e in ew]))
            if "rec" in ep:
                for g in range(2):
                    for nm in ep["rec"][g]:
                        assert _same(ep["rec"][g][nm], ew[g]["rec"][0][nm]), f"{case}: recorder {nm} differs"
            sp = per.episode_stats()
            sw = [w.episode_stats() for w in whole]
            assert sp[0] == sw[0][0] + sw[1][0] and sp[2] == sw[0][2] + sw[1][2], f"{case}: episode counts differ"
            assert abs(sp[1] - sw[0][1] - sw[1][1]) <= 1e-9 * max(1.0, abs(sp[1]))  # sums in another atomic order
    assert (per.get("ep_idx") >= 3).all(), "every env must have run through auto-resets"
    if whole_b is not whole:
        print(f"{case}: twin vs whole-batch tier from the same state, max d obs / (1 + |obs|) = {d_batch:.3e}")
    for eng in {id(e): e for e in [per] + whole + whole_b}.values():
        eng.close()


def test_f64_model_step_per_env_equals_whole_batch(E):
    """env_layer = 0: b747_model_step of a per-env handle against one whole-batch handle per parameter set."""
    n = 512
    sizes, starts = [256, 256], [0, 256]
    kw = dict(dtype=E.F64, env_layer=False, export_signals=True, seed=4)
    per = E.BatchEngine(n_envs=n, **kw)
    whole = [E.BatchEngine(n_envs=256, env_id_offset=starts[g], **kw) for g in range(2)]
    psets = [_param_set(per, g) for g in range(2)]
    for g in range(2):
        for nm, v in psets[g].items():
            whole[g].set_param(nm, v)
    for nm in NAMES:
        vals = _concat([np.tile(psets[g][nm], (sizes[g], 1)) for g in range(2)])
        per.set_env_param(nm, vals if E_N(nm) > 1 else vals[:, 0])
    for eng in [per] + whole:
        eng.reset()
        eng.model_initialize()
    for k in range(6):
        for eng in [per] + whole:
            eng.model_step(50)
        fp, fw = _fields(per), [_fields(w) for w in whole]
        for nm in fp:
            assert _same(fp[nm], _concat([f[nm] for f in fw])), f"model step: field {nm} differs after block {k}"
    assert not np.array_equal(fw[0]["h"], fw[1]["h"]), "the two parameter sets must fly differently"


class _Models:
    """Oracle models of a model-stepping handle, with OracleBatch's gather / ticks (test_gpu_parity._field_ratios)."""

    def __init__(self, models):
        self.m = models

    def gather(self, name, idx=0):
        return np.array([np.atleast_1d(m.get(name))[idx] for m in self.m])

    def ticks(self):
        return np.array([m.tick for m in self.m], np.int64)


@pytest.mark.parametrize("per_env", [True, False])
def test_model_step_tunables_match_oracle(E, per_env):
    """env_layer = 0 with use_PID_SS = use_PID_CS = 1, so that both gain sets act: b747_model_step with every tunable
    away from its default -- per env (k_model_step64<true>, values inside tuned_ranges, g set for the batch) or by
    set_param (k_model_step64<false>, tuned_params) -- against oracle models given the same values: the 16 states,
    every exported signal and the tick of every env at 1e-9 after every 20 of 400 model steps."""
    from oracle import oracle as O
    from test_gpu_parity import _field_ratios, tuned_params, tuned_ranges
    O.build()
    n = 256
    rng = np.random.default_rng(6)
    tp = tuned_params(O)
    if per_env:
        vals = {nm: lo + (hi - lo) * rng.uniform(size=(n, len(lo))) for nm, (lo, hi) in tuned_ranges(O).items()}
        vals["g"] = np.tile(tp["g"], (n, 1))
    else:
        vals = {nm: np.tile(v, (n, 1)) for nm, v in tp.items()}
    s0 = np.stack([np.zeros(n), rng.uniform(3000, 10000, n), rng.uniform(200, 260, n), rng.uniform(-5, 5, n),
                   rng.uniform(-0.05, 0.05, n), np.zeros(n)], axis=1)
    hzh, vzh = s0[:, 1] + rng.uniform(-300, 300, n), rng.uniform(-0.1, 0.1, n)
    eng = E.BatchEngine(n_envs=n, dtype=E.F64, env_layer=False, export_signals=True, seed=4)
    for nm, v in vals.items():
        if per_env and nm != "g":
            eng.set_env_param(nm, v if E_N(nm) > 1 else v[:, 0])
        else:
            eng.set_param(nm, v[0])
    eng.set_param("use_PID_SS", 1.0)
    eng.reset()
    for k, nm in enumerate(("state0_x", "state0_y", "state0_Vx", "state0_Vy", "state0_vartheta", "state0_wz")):
        eng.set(nm, s0[:, k])
    eng.model_initialize()
    eng.set("h_zh", hzh)
    eng.set("vartheta", vzh)
    eng.set("deltaz", np.zeros(n))
    eng.set("flags", (eng.get("flags").astype(np.int64) | 4).astype(np.float64))   # use_PID_CS >= 1 (core/model.py)
    models = [O.CModel() for _ in range(n)]
    for i, m in enumerate(models):
        for nm, v in vals.items():
            m.set(nm, v[i] if len(v[i]) > 1 else v[i][0])
        m.set("state0", s0[i])
        m.initialize()
        for nm, v in (("h_zh", hzh[i]), ("vartheta", vzh[i]), ("deltaz", 0.0), ("use_PID_SS", 1.0), ("use_PID_CS", 1.0)):
            m.set(nm, v)
    ob = _Models(models)
    ratios = {}
    for _ in range(20):
        eng.model_step(20)
        for m in models:
            m.step(20)
        _field_ratios(eng, ob, ratios)
    print("model step, worst fields (deviation / bar):", sorted(ratios.items(), key=lambda kv: -kv[1])[:4])
    assert all(v <= 1.0 for v in ratios.values()), {k: v for k, v in ratios.items() if not v <= 1.0}
    assert np.abs(ob.gather("vartheta_zh")).min() > 0 and np.abs(ob.gather("U_com_PID")).min() > 0  # both loops act
    eng.close()


ROUTING_SCRIPT = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from torch.profiler import ProfilerActivity, profile
from b747_rl_ctrl_b200 import engine as E

def names(eng, step, path):
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        eng.synchronize()
    prof.export_chrome_trace(path)
    with open(path) as f:
        ev = json.load(f)["traceEvents"]
    return [e["name"] for e in ev if e.get("cat") == "kernel" and ("k_env_step" in e["name"] or "k_model_step" in e["name"])]

out = {}
cases = {"canonical": dict(), "tier1": dict(obs_type=1, ctrl_mode=1, action_max=1.0),
         "tier2": dict(rew_type=2, ctrl_type=2, reset_ref_mode=2), "tier3": dict(export_signals=True),
         "f64": dict(dtype=E.F64)}
for tag, kw in cases.items():
    eng = E.BatchEngine(n_envs=4096, seed=2, **kw)
    eng.reset()
    a = np.zeros(4096, eng.np_dtype)
    out[tag + "-batch"] = names(eng, lambda: eng.step_host(a), sys.argv[2] + "/b.json")
    eng.set_env_param("m0", np.full(4096, eng.get_param("m0")))
    out[tag] = names(eng, lambda: eng.step_host(a), sys.argv[2] + "/p.json")
    eng.close()
eng = E.BatchEngine(n_envs=256, dtype=E.F64, env_layer=False)
eng.set_env_param_range("PID_SS", [0.1] * 4, [0.2] * 4)
out["model"] = names(eng, lambda: eng.model_step(1), sys.argv[2] + "/m.json")
# test_entering_per_env_mode_mid_run's handles: per-env mode entered after an auto-reset, in the middle of an episode
for tag, dt in (("midrun", E.F32), ("midrun-f64", E.F64)):
    eng = E.BatchEngine(n_envs=512, dtype=dt, seed=9, sample_time=0.1, tk=2.0)
    eng.reset()
    a = np.zeros(512, eng.np_dtype)
    for _ in range(29):
        eng.step_host(a)
    out[tag + "-batch"] = names(eng, lambda: eng.step_host(a), sys.argv[2] + "/r.json")
    eng.set_env_param("Iz", np.full(512, 6.0e7))
    eng.set_env_param_range("P", [2.5e5], [3.0e5])
    out[tag] = names(eng, lambda: eng.step_host(a), sys.argv[2] + "/s.json")
    eng.close()
print(json.dumps(out))
"""


def test_routing(E, tmp_path):
    """One profiled launch per case, in a child process (its own profiler session): the twins' template arguments,
    tier 0 for a canonical handle without per-env mode, and the switch of test_entering_per_env_mode_mid_run's handles
    (plain kernel after an auto-reset, twin once per-env values and a range arrive mid-episode)."""
    import json
    import subprocess
    want = {
        "canonical-batch": "k_env_step32<0, 4, false, false>",
        "canonical": "k_env_step32<5, -1, false, false>",
        "tier1": "k_env_step32<5, -1, false, false>",
        "tier2": "k_env_step32<6, -1, false, false>",
        "tier3": "k_env_step32<7, -1, false, false>",
        "f64-batch": "k_env_step64<false>",
        "f64": "k_env_step64<true>",
        "model": "k_model_step64<true>",
        "midrun-batch": "k_env_step32<0, 4, false, false>",
        "midrun": "k_env_step32<5, -1, false, false>",
        "midrun-f64-batch": "k_env_step64<false>",
        "midrun-f64": "k_env_step64<true>",
    }
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", ROUTING_SCRIPT, os.path.dirname(HERE), str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    for tag, name in want.items():
        assert len(got[tag]) == 1 and name in got[tag][0], (tag, got[tag])


# ---- draws ---------------------------------------------------------------------------------------------------------
def _u53(L, seed, env, epi, draw):
    ctr = (ctypes.c_uint32 * 4)(env & 0xffffffff, env >> 32, epi, draw >> 1)
    key = (ctypes.c_uint32 * 2)(seed & 0xffffffff, seed >> 32)
    w = (ctypes.c_uint32 * 4)()
    L.b747_philox4x32(ctr, key, w)
    a, b = w[2 * (draw & 1)] >> 5, w[2 * (draw & 1) + 1] >> 6
    return (a * 67108864.0 + b) * (1.0 / 9007199254740992.0)


RANGES = {"m0": (2.4e5, 3.6e5), "Iz": (2.0e7, 3.5e7), "P": (3.0e5, 4.0e5), "S": (480.0, 560.0), "c_": (7.5, 9.0),
          "PID_SS": ([-3, 0.1, -1, 10], [-1, 0.5, -0.2, 40]), "PID_CS": ([0.001, 1e-5, 0.01, 5], [0.01, 1e-4, 0.1, 20])}


def _expected(L, seed, env_ids, epis, name):
    lo, hi = (np.atleast_1d(np.asarray(x, np.float64)) for x in RANGES[name])
    out = np.empty((len(env_ids), len(lo)))
    for k, (e, p) in enumerate(zip(env_ids, epis)):
        for j in range(len(lo)):
            out[k, j] = lo[j] + (hi[j] - lo[j]) * _u53(L, seed, int(e), int(p), 32 + ROW0[name] + j)
    return out if len(lo) > 1 else out[:, 0]


def _check_draws(E, eng, L, seed, off, envs=None):
    epi = eng.get("ep_idx").astype(np.int64) - 1
    envs = np.arange(eng.n_envs) if envs is None else np.asarray(envs)
    for nm in NAMES:
        got = eng.get_env_param(nm).cpu().numpy()[envs]
        want = _expected(L, seed, envs + off, epi[envs], nm)
        assert _same(got, want), f"{nm}: drawn values differ from lo + (hi - lo) u"


@pytest.mark.parametrize("f64", [False, True])
def test_draws(E, f64):
    from b747_rl_ctrl_b200 import _lib
    L = _lib.load()
    n, seed, off = 600, 0x1234567890AB, 70
    kw = dict(n_envs=n, dtype=E.F64 if f64 else E.F32, seed=seed, env_id_offset=off, disturbance_mode=E.DIST_AERO,
              obs_type=1, **K5)
    eng, ref = E.BatchEngine(**kw), E.BatchEngine(**kw)
    for nm, (lo, hi) in RANGES.items():
        eng.set_env_param_range(nm, lo, hi)
    eng.reset()
    ref.reset()
    _check_draws(E, eng, L, seed, off)
    rng = np.random.default_rng(1)
    for k in range(45):  # two auto-resets of every env
        a = rng.uniform(-1, 1, n).astype(eng.np_dtype)
        o1, r1, d1 = eng.step_host(a)
        ref.step_host(a)
        if k % 11 == 10:
            _check_draws(E, eng, L, seed, off)
    _check_draws(E, eng, L, seed, off)
    # the episode draws are those of a handle without ranges
    f, g = _fields(eng), _fields(ref)
    for nm in ("vref", "href", "ep_idx", "state0_x", "state0_y", "state0_Vx", "state0_Vy", "state0_wz", "aerr0", "aerr1",
               "aerr2", "aerr3", "aerr4", "tick"):
        if nm in f:
            assert _same(f[nm], g[nm]), f"episode draw {nm} changed by the parameter ranges"
    # masked reset: only masked envs redraw
    import torch
    before = {nm: eng.get_env_param(nm).cpu().numpy() for nm in NAMES}
    mask = (np.arange(n) % 3 == 0).astype(np.uint8)
    mask_d, unmask_d = torch.from_numpy(mask).cuda(), torch.from_numpy(1 - mask).cuda()
    torch.cuda.synchronize()  # the masks are read on the handle's stream
    eng.reset(mask=mask_d)
    eng.synchronize()
    for nm in NAMES:
        now = eng.get_env_param(nm).cpu().numpy()
        assert _same(now[mask == 0], before[nm][mask == 0]), f"{nm}: an unmasked env redrew"
        assert not np.array_equal(now[mask == 1], before[nm][mask == 1])
    _check_draws(E, eng, L, seed, off, np.nonzero(mask)[0])
    # explicit episodes and loads leave the values alone
    before = {nm: eng.get_env_param(nm).cpu().numpy() for nm in NAMES}
    ep = E.episode([0, 5000, 200, 0, 0, 0], vref=0.05)
    eng.reset_to([ep] * n)
    eng.reset_to([ep] * n, mask=unmask_d)
    blob = ref.save_state()
    eng.load_state(blob)
    eng.synchronize()
    for nm in NAMES:
        assert _same(eng.get_env_param(nm), before[nm]), f"{nm}: changed by reset_to / load_state"
    eng.close()
    ref.close()


# ---- float64 oracle ------------------------------------------------------------------------------------------------
ORACLE_FAMILIES = {  # engine / oracle keywords, engine-only keywords, family of DESIGN.md 4.2 (test_gpu_parity)
    "canonical": (dict(), None, "K10"),                                                     # tier-1 twin
    "speed-addproc": (dict(obs_type=1, ctrl_mode=1, action_max=1.0), None, "speed_addproc"),  # PID_SS feeds the elevator
    "quality-semi-hybrid": (dict(rew_type=2, ctrl_type=2, reset_ref_mode=2), None, "quality_semimanual"),  # tier 2, PID_CS
    "canonical-full": (dict(), dict(export_signals=True, track_transfer=True, record_capacity=16), "K10"),  # tier-3 twin
}


@pytest.mark.parametrize("fam", list(ORACLE_FAMILIES))
@pytest.mark.parametrize("f64", [False, True])
def test_against_oracle(E, fam, f64):
    """All 13 per-env components drawn at every reset (m0, Iz +-20 %, P, S, c_ +-10 %, every PID_SS / PID_CS component
    0.7-1.3 x its default) and g set for the whole batch.  The oracle computes each env's values itself (lo + (hi - lo) u
    from its own Philox, episode index counted from its own done flags); the handle's get_env_param equals them bit for
    bit after every reset.  512 envs, five 10-step episodes.  float64 with signals: observations, rewards, the 16
    states, every exported signal and the tick at test_gpu_parity's bars; f32 twins: the family bounds of DESIGN.md 4.2
    inside the flight envelope.  The measured maxima are printed."""
    from oracle import oracle as O
    from test_gpu_parity import (F64_OBS_TOL, F64_REW_TOL, FAMILY_BOUNDS, _assert_bound, _f32_bound_rollout,
                                 _rollout_compare, tuned_params, tuned_ranges)
    O.build()
    kw, ekw, bound = ORACLE_FAMILIES[fam]
    kw = dict(sample_time=0.05, tk=0.5, **kw)
    params, ranges = {"g": tuned_params(O)["g"]}, tuned_ranges(O)
    n, steps = 512, 50
    if f64:
        wo, wr, nd, eng = _rollout_compare(E, O, E.F64, n, steps, kw, 9, F64_OBS_TOL, F64_REW_TOL, fields=True, ekw=ekw,
                                           params=params, ranges=ranges)
        print(f"oracle {fam} f64: max |d obs| {wo:.3e}, max |d rew| {wr:.3e}")
        eng.close()
    else:
        res = _f32_bound_rollout(E, O, n, steps, kw, 9, ekw=ekw, params=params, ranges=ranges)
        _assert_bound(f"oracle {fam} twin", res, *FAMILY_BOUNDS[bound])
        nd = res["n_done"]
    assert nd == n * steps // 10


@pytest.mark.parametrize("per_env", [False, True])
def test_tunables_survive_hybrid_resets(E, per_env):
    """A HYBRID reset of the reference re-creates its Model with the default gains and thrust (Controller._init_model);
    the kernels keep the handle's tunables -- set_param values, or set_env_param values of every env -- across every
    reset.  They read back unchanged after three episodes, the float64 run matches the oracle given them again after
    each of its HYBRID resets (reapply_after_hybrid_reset), and it does not match an oracle left at its defaults."""
    from oracle import oracle as O
    from test_gpu_parity import F64_OBS_TOL, F64_REW_TOL, _rollout_compare, tuned_params, tuned_ranges
    O.build()
    kw = dict(rew_type=2, ctrl_type=2, reset_ref_mode=2, sample_time=0.05, tk=0.5)
    n = 256
    rng = np.random.default_rng(3)
    vals = {nm: lo + (hi - lo) * rng.uniform(size=(n, len(lo))) for nm, (lo, hi) in tuned_ranges(O).items()}
    params = None if per_env else tuned_params(O)

    def give(eng, tun):
        for nm, v in vals.items():
            eng.set_env_param(nm, v if E_N(nm) > 1 else v[:, 0])
            tun.set_env_param(nm, v)

    def run(reapply):
        return _rollout_compare(E, O, E.F64, n, 30, kw, 9, F64_OBS_TOL, F64_REW_TOL, fields=True, params=params,
                                at_step={0: give} if per_env else None, reapply_hybrid=reapply)

    _, _, nd, eng = run(True)
    assert nd == 3 * n
    if per_env:
        for nm, v in vals.items():
            assert _same(eng.get_env_param(nm).cpu().numpy().reshape(n, -1), v), f"{nm} changed by a HYBRID reset"
    else:
        for nm, v in params.items():
            assert _same(np.atleast_1d(eng.get_param(nm, len(v))), v), f"{nm} changed by a HYBRID reset"
    eng.close()
    with pytest.raises(AssertionError):
        run(False)


@pytest.mark.parametrize("f64", [False, True])
def test_entering_per_env_mode_mid_run(E, f64):
    """A canonical K = 10 handle steps through an auto-reset on its plain kernel (f32: tier 0, whose auto-reset writes
    only the lean state groups, so the twin then reads general groups last written by b747_reset; f64:
    k_env_step64<false>) and takes per-env values of every name, and ranges of P, PID_SS and PID_CS, in the middle of its
    second episode.  The oracle takes the same values at the same step and draws the ranged ones at its later resets.
    Two more episodes against the oracle -- f32: the K10 bound of DESIGN.md 4.2, f64: every field at 1e-9.  That the
    plain kernel runs before the switch and the twin after it is checked by kernel name in test_routing (one profiler
    session per process)."""
    from oracle import oracle as O
    from test_gpu_parity import (F64_OBS_TOL, F64_REW_TOL, FAMILY_BOUNDS, _assert_bound, _f32_bound_rollout,
                                 _rollout_compare, tuned_ranges)
    O.build()
    kw = dict(sample_time=0.1, tk=2.0)   # 20-step episodes
    n, switch, steps = 512, 30, 70
    rng = np.random.default_rng(8)
    ranges = tuned_ranges(O)
    vals = {nm: lo + (hi - lo) * rng.uniform(size=(n, len(lo))) for nm, (lo, hi) in ranges.items()}

    def enter(eng, tun):
        for nm, v in vals.items():
            eng.set_env_param(nm, v if E_N(nm) > 1 else v[:, 0])
            tun.set_env_param(nm, v)
        for nm in ("P", "PID_SS", "PID_CS"):
            eng.set_env_param_range(nm, *ranges[nm])
            tun.set_range(nm, *ranges[nm])

    if f64:
        wo, wr, nd, eng = _rollout_compare(E, O, E.F64, n, steps, kw, 9, F64_OBS_TOL, F64_REW_TOL, fields=True,
                                           at_step={switch: enter})
        eng.close()
        print(f"f64 entering per-env mode at step {switch}: max |d obs| {wo:.3e}, max |d rew| {wr:.3e}")
    else:
        res = _f32_bound_rollout(E, O, n, steps, kw, 9, at_step={switch: enter})
        _assert_bound(f"tier 0 -> twin at step {switch}", res, *FAMILY_BOUNDS["K10"])
        nd = res["n_done"]
    assert nd == 3 * n


# ---- API -----------------------------------------------------------------------------------------------------------
def test_argument_checks_change_nothing(E):
    import torch
    eng = E.BatchEngine(n_envs=100, seed=3)
    L, h = eng._L, eng._h
    dp = ctypes.POINTER(ctypes.c_double)
    arr = lambda *v: (ctypes.c_double * len(v))(*v)
    bad = [("mass", arr(1.0), arr(2.0), 1), ("m0", arr(1.0, 2.0), arr(2.0, 3.0), 2), ("m0", arr(math.inf), arr(2.0), 1),
           ("m0", arr(math.nan), arr(2.0), 1), ("P", arr(3.0), arr(2.0), 1), ("m0", arr(0.0), arr(2.0), 1),
           ("Iz", arr(-1.0), arr(2.0), 1), ("S", arr(0.0), arr(1.0), 1), ("c_", arr(-2.0), arr(1.0), 1),
           ("PID_SS", arr(1, 1, 1, 1), arr(2, 2, 0, 2), 4), ("g", arr(1.0), arr(2.0), 1), ("use_RP", arr(0.0), arr(1.0), 1)]
    for nm, lo, hi, nc in bad:
        assert L.b747_set_env_param_range(h, nm.encode(), ctypes.cast(lo, dp), ctypes.cast(hi, dp), nc) == -1, nm
    assert L.b747_set_env_param_range(h, b"m0", ctypes.cast(arr(1.0), dp), None, 1) == -1
    v = torch.zeros(101, dtype=torch.float64, device="cuda")
    idx = torch.zeros(11, dtype=torch.int32, device="cuda")
    assert L.b747_set_env_param(h, b"m0", ctypes.c_void_p(v.data_ptr() + 4), None, 10) == -1
    assert L.b747_set_env_param(h, b"m0", ctypes.c_void_p(v.data_ptr()), ctypes.c_void_p(idx.data_ptr() + 2), 10) == -1
    assert L.b747_set_env_param(h, b"m0", ctypes.c_void_p(v.data_ptr()), None, 101) == -1
    assert L.b747_set_env_param(h, b"PID", ctypes.c_void_p(v.data_ptr()), None, 10) == -1
    assert L.b747_get_env_param(h, b"m0", None, 10, ctypes.c_void_p(v.data_ptr() + 4)) == -1
    # nothing changed: not in per-env mode, the canonical tier still runs and a reset draws nothing
    m0 = eng.get_param("m0")
    eng.reset()
    assert (eng.get_env_param("m0").cpu().numpy() == m0).all()
    assert (eng.get_env_param("PID_SS").cpu().numpy() == eng.get_param("PID_SS", 4)).all()
    eng.close()


def test_scatter_gather_and_broadcast(E):
    import torch
    n = 300
    eng = E.BatchEngine(n_envs=n, seed=3)
    base = eng.get_param("PID_SS", 4)
    idx = np.array([5, -1, 299, 300, 17, 1 << 30], np.int32)
    vals = np.arange(24, dtype=np.float64).reshape(6, 4) + 1.0
    eng.set_env_param("PID_SS", vals, idx)
    got = eng.get_env_param("PID_SS").cpu().numpy()
    want = np.tile(base, (n, 1))
    for k, i in enumerate(idx):
        if 0 <= i < n:
            want[i] = vals[k]
    assert _same(got, want)
    g = eng.get_env_param("PID_SS", torch.from_numpy(idx).cuda()).cpu().numpy()
    for k, i in enumerate(idx):
        assert _same(g[k], want[i]) if 0 <= i < n else np.isnan(g[k]).all()
    # set_param in per-env mode: the batch value and every env's value of that name
    eng.set_param("m0", 3.0e5)
    assert eng.get_param("m0") == 3.0e5
    assert (eng.get_env_param("m0").cpu().numpy() == 3.0e5).all()
    assert _same(eng.get_env_param("PID_SS"), want), "set_param of another name must leave PID_SS alone"
    eng.set_param("PID_SS", base)
    assert (eng.get_env_param("PID_SS").cpu().numpy() == base).all()
    # ... and it steps like a whole-batch handle with that value
    ref = E.BatchEngine(n_envs=n, seed=3)  # the same kernel (the tier-1 twin) with m0 written env by env
    ref.set_env_param("m0", np.full(n, 3.0e5))
    eng.reset(); ref.reset()
    a = np.random.default_rng(2).uniform(-1, 1, n).astype(np.float32)
    for _ in range(30):
        assert _same(eng.step_host(a)[0], ref.step_host(a)[0])
    eng.close(); ref.close()


@pytest.mark.parametrize("f64", [False, True])
def test_fork_recipe(E, f64):
    """64 sources -> 64 x 8 candidates: blob and per-env parameters copied with the same index arrays; every candidate
    repeats its source bit for bit until the source's episode ends."""
    import torch
    dt = E.F64 if f64 else E.F32
    src = E.BatchEngine(n_envs=64, dtype=dt, seed=21, **K5)
    for nm, (lo, hi) in RANGES.items():
        src.set_env_param_range(nm, lo, hi)
    src.reset()
    rng = np.random.default_rng(4)
    for _ in range(7):
        src.step_host(rng.uniform(-1, 1, 64).astype(src.np_dtype))
    blob = src.save_state()
    bidx = torch.arange(512, dtype=torch.int32, device="cuda") // 8
    cand = E.BatchEngine(n_envs=512, dtype=dt, seed=21, **K5)
    cand.load_state(blob, blob_indices=bidx)
    for nm in NAMES:
        cand.set_env_param(nm, src.get_env_param(nm, bidx))
    alive = np.ones(64, bool)
    for _ in range(25):
        a = rng.uniform(-1, 1, 64).astype(src.np_dtype)
        o, r, d = src.step_host(a)
        oc, rc, dc = cand.step_host(np.repeat(a, 8))
        for j in np.nonzero(alive)[0]:
            assert _same(oc[8 * j:8 * j + 8], np.tile(o[j], (8, 1))) and _same(rc[8 * j:8 * j + 8], np.full(8, r[j]))
        alive &= ~d.astype(bool)
    assert not alive.any()
    src.close(); cand.close()


def test_vec_env_param_ranges(E):
    from b747_rl_ctrl_b200.vec_env import B747VecEnv
    env = B747VecEnv(256, tk=1.0, param_ranges={"m0": (2.5e5, 3.5e5), "PID_SS": ([-3, 0.1, -1, 10], [-1, 0.5, -0.2, 40])})
    env.reset()
    m0a = env.get_env_param("m0")
    assert m0a.shape == (256,) and len(np.unique(m0a)) == 256 and ((m0a >= 2.5e5) & (m0a <= 3.5e5)).all()
    for _ in range(25):  # one auto-reset of every env
        env.step(np.zeros((256, 1), np.float32))
    m0b = env.get_env_param("m0")
    assert (m0b != m0a).all()
    assert _same(m0b, env.engine.get_env_param("m0"))
    assert env.get_env_param("PID_SS").shape == (256, 4)
    env.close()
