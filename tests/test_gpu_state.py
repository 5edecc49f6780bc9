"""Save, restore and fork per-env state on the GPU (b747_save_state / b747_load_state, BatchEngine.save_state /
load_state, B747VecEnv.get_state / set_state).

  * replay: step, save every env, step T seeded steps across auto-resets, load, step the same T again -- outputs, packed
    records, every per-env field, last_episode(), transfer metrics and recorder rows must repeat bit for bit, for every
    f32 kernel tier at multi-tile scale, for float64 with the evaluation features and for raw float64 model stepping;
  * subsets and forks: a ragged index list loaded into other positions of a fresh handle, and 64 states fanned out
    into 64 x 512 candidates, reproduce their sources until the first done, and envs not named stay untouched;
  * a blob saved on the full f32 kernel tier moves the loading handle there;
  * blobs of another dtype or configuration, corrupted headers and out-of-range indices are refused without a fault.
"""
import ctypes
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
from test_gpu_scale import _profiled, _template_args  # noqa: E402

pytestmark = pytest.mark.gpu

N_BIG = (1 << 18) + 77
T = 40        # replayed steps: every family finishes episodes inside them
PHASES = 4    # episode phases: env i is reset once more after step i % PHASES of the warm-up

K1 = dict(sample_time=0.01, tk=0.3)     # 30-step episodes, the TMA-staged kernel
K10 = dict(sample_time=0.1, tk=1.0)     # 10-step episodes
K5 = dict(sample_time=0.05, tk=1.0)     # 20-step episodes
TRACE = dict(export_signals=True, track_transfer=True, record_capacity=12)
FAMILIES = {
    "f32-T0-K1": dict(n=N_BIG, kw=K1),
    "f32-T0-K10": dict(n=N_BIG, kw=K10),
    "f32-T1": dict(n=N_BIG, kw=dict(obs_type=1, ctrl_mode=1, action_max=1.0, **K5)),
    "f32-T2": dict(n=N_BIG, kw=dict(rew_type=2, ctrl_type=2, reset_ref_mode=2, **K5)),
    "f32-T3": dict(n=N_BIG, kw=dict(**K5, **TRACE)),
    "f64": dict(n=4096, f64=True, kw=dict(**K5, **TRACE)),
}


def _bits(x):
    x = x.cpu().numpy() if hasattr(x, "cpu") else np.asarray(x)
    return np.ascontiguousarray(x).view(np.uint8)


def _same(a, b):
    return a.shape == b.shape and np.array_equal(_bits(a), _bits(b))


@pytest.fixture(scope="module")
def E():
    import torch
    assert torch.cuda.is_available()
    from b747_rl_ctrl_b200 import engine
    return engine


def _make(E, n, f64=False, seed=17, **kw):
    return E.BatchEngine(n_envs=n, dtype=E.F64 if f64 else E.F32, seed=seed, **kw)


def _spread(E, eng, steps=PHASES + 3):
    """Reset, then step with seeded actions, resetting env i once more after step i % PHASES: episode phases differ."""
    import torch
    dev = torch.device("cuda")
    n = eng.n_envs
    eng.reset()
    acts = torch.from_numpy(np.random.default_rng(5).uniform(-1, 1, (steps, n)).astype(eng.np_dtype)).to(dev)
    _, obs, rew, done, term = eng.alloc_io(terminal_obs=True)
    phase = torch.arange(n, device=dev) % PHASES
    masks = [(phase == k).to(torch.uint8) for k in range(PHASES)]
    torch.cuda.synchronize()
    for k in range(steps):
        eng.step(acts[k], obs, rew, done, term)
        if k < PHASES:
            eng.reset(mask=masks[k])
    eng.synchronize()


def _fields(E, eng):
    out = {}
    for f in eng.field_names():
        try:
            out[f] = eng.get(f)
        except E.B747Error:
            pass   # not carried by this handle
    return out


def _run(E, eng, acts, packed):
    """T steps; f32 handles alternate between b747_step and b747_step_packed.  Everything observable, on the host."""
    import torch
    n, od = eng.n_envs, eng.obs_dim
    eng.episode_stats()   # zero the accumulators (they are not part of a blob)
    _, obs, rew, done, term = eng.alloc_io(terminal_obs=True)
    h = dict(obs=[], rew=[], done=[], term=[], rec=[], bits=[])
    if packed:
        rec = torch.empty(n, eng.record_floats, device="cuda")
        bits = torch.empty((n + 31) // 32, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    for k in range(len(acts)):
        if packed and k % 2:
            eng.step_packed(acts[k], rec, bits)
            eng.synchronize()
            h["rec"].append(rec.cpu().numpy())
            h["bits"].append(bits.cpu().numpy())
        else:
            eng.step(acts[k], obs, rew, done, term)
            eng.synchronize()
            for key, v in (("obs", obs), ("rew", rew), ("done", done), ("term", term)):
                h[key].append(v.cpu().numpy())
    out = {k: np.stack(v) for k, v in h.items() if v}
    out.update(_observe(E, eng))
    out["stats"] = eng.episode_stats()
    return out


def _observe(E, eng):
    """Every per-env field, last_episode(), transfer metrics (both modes) and a few envs' recorder rows."""
    n = eng.n_envs
    out = dict(fields=_fields(E, eng), last_episode=eng.last_episode())
    if eng.cfg.track_transfer:
        out["metrics"] = {(w, f): eng.transfer_metrics(w, f) for w in ("SS", "CS") for f in (True, False)}
    if eng.cfg.record_capacity:
        out["recorder"] = {i: eng.recorder_read(i) for i in (0, 1234 % n, n - 1)}
    return out


def _diffs(a, b):
    bad = []
    for k in ("obs", "rew", "done", "term", "rec", "bits"):
        if k in a and not _same(a[k], b[k]):
            bad.append(k)
    for f in a["fields"]:
        if not _same(a["fields"][f], b["fields"][f]):
            bad.append("field " + f)
    for i in (0, 1):
        if not _same(a["last_episode"][i], b["last_episode"][i]):
            bad.append("last_episode")
    for key, v in a.get("metrics", {}).items():
        if not _same(v, b["metrics"][key]):
            bad.append(f"metrics {key}")
    for i, r in a.get("recorder", {}).items():
        for key, v in r.items():
            if not _same(v, b["recorder"][i][key]):
                bad.append(f"recorder env {i} {key}")
    return bad


@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_replay_after_load_is_exact(E, family):
    import torch
    c = FAMILIES[family]
    eng = _make(E, c["n"], f64=c.get("f64", False), **c["kw"])
    _spread(E, eng)
    blob = eng.save_state()
    assert blob.numel() == eng.state_bytes()
    saved = _observe(E, eng)
    acts = torch.from_numpy(np.random.default_rng(11).uniform(-1, 1, (T, eng.n_envs)).astype(eng.np_dtype)).cuda()
    packed = not c.get("f64", False)
    a = _run(E, eng, acts, packed)
    eng.load_state(blob)
    bad = _diffs(saved, _observe(E, eng))   # state that the next step overwrites before reading it is restored too
    assert not bad, f"{family}: not restored by the load: {bad[:8]}"
    b = _run(E, eng, acts, packed)
    n_done = int(a["done"].sum()) + (int(np.unpackbits(a["bits"].view(np.uint8)).sum()) if packed else 0)
    assert n_done >= eng.n_envs, "the replay must cross auto-resets"
    bad = _diffs(a, b)
    assert not bad, f"{family}: differs after load: {bad[:8]}"
    assert len(a["fields"]) >= (30 if packed else 80)
    sa, sb = a["stats"], b["stats"]
    assert sa[0] == sb[0] and sa[2] == sb[2] and sa[0] > 0
    assert abs(sa[1] - sb[1]) <= 1e-12 * abs(sa[1]) and abs(sa[3] - sb[3]) <= 1e-12 * abs(sa[3])
    eng.close()


def test_replay_raw_model_stepping_f64(E):
    """env_layer = 0: b747_model_step with per-step deltaz edits repeats every field after a load."""
    n = 4096
    eng = _make(E, n, f64=True, env_layer=False, **TRACE)
    eng.model_initialize()
    rng = np.random.default_rng(3)
    eng.set("deltaz", rng.uniform(-0.1, 0.1, n))
    eng.model_step(7)
    blob = eng.save_state()
    dz = rng.uniform(-0.1, 0.1, (12, n))

    def run():
        hist = []
        for k in range(len(dz)):
            eng.set("deltaz", dz[k])
            eng.model_step(3)
            hist.append(_fields(E, eng))
        return hist

    a = run()
    eng.load_state(blob)
    b = run()
    for k in range(len(dz)):
        bad = [f for f in a[k] if not _same(a[k][f], b[k][f])]
        assert not bad, f"step {k}: {bad[:8]}"
    assert not np.array_equal(a[0]["h"], a[-1]["h"])
    eng.close()


def _outputs(E, eng, acts):
    import torch
    _, obs, rew, done, term = eng.alloc_io(terminal_obs=True)
    h = dict(obs=[], rew=[], done=[], term=[])
    torch.cuda.synchronize()
    for k in range(len(acts)):
        eng.step(acts[k], obs, rew, done, term)
        eng.synchronize()
        for key, v in (("obs", obs), ("rew", rew), ("done", done), ("term", term)):
            h[key].append(v.cpu().numpy())
    return {k: np.stack(v) for k, v in h.items()}


def _until_first_done(a, ia, b, ib):
    """Rows ia of history a equal rows ib of history b (bit for bit) up to each env's first done; the post-reset
    observation of that step is excluded (resets draw from the env's own id).  Returns how many envs finished."""
    done = a["done"][:, ia].astype(bool)
    finished = 0
    for j in range(len(ia)):
        d = np.flatnonzero(done[:, j])
        last = d[0] if len(d) else len(done) - 1
        finished += bool(len(d))
        for key in ("rew", "done", "term"):
            assert _same(a[key][:last + 1, ia[j]], b[key][:last + 1, ib[j]]), (key, ia[j], ib[j])
        assert _same(a["obs"][:last, ia[j]], b["obs"][:last, ib[j]]), ("obs", ia[j], ib[j])
    return finished


@pytest.mark.parametrize("f64", [False, True], ids=["f32", "f64"])
def test_subset_into_other_positions(E, f64):
    import torch
    n, m = 5000, 777
    kw = dict(**K5)
    src = _make(E, n, f64=f64, **kw)
    _spread(E, src)
    rng = np.random.default_rng(8)
    idx_src = np.sort(rng.choice(n, m, replace=False)).astype(np.int32)     # ragged, non-contiguous
    idx_dst = rng.choice(n, m, replace=False).astype(np.int32)
    blob = src.save_state(idx_src)
    assert blob.numel() == src.state_bytes(m)
    dst, ctl = _make(E, n, f64=f64, **kw), _make(E, n, f64=f64, **kw)
    dst.reset()
    ctl.reset()
    dst.load_state(blob, indices=torch.from_numpy(idx_dst).cuda())
    a_src = rng.uniform(-1, 1, (T, n)).astype(src.np_dtype)
    a_ctl = rng.uniform(-1, 1, (T, n)).astype(src.np_dtype)
    a_dst = a_ctl.copy()
    a_dst[:, idx_dst] = a_src[:, idx_src]
    hs, hd, hc = (_outputs(E, e, torch.from_numpy(a).cuda()) for e, a in ((src, a_src), (dst, a_dst), (ctl, a_ctl)))
    assert _until_first_done(hs, idx_src, hd, idx_dst) == m
    others = np.setdiff1d(np.arange(n), idx_dst)
    for key in hd:
        assert _same(hd[key][:, others], hc[key][:, others]), key
    for e in (src, dst, ctl):
        e.close()


@pytest.mark.parametrize("f64", [False, True], ids=["f32", "f64"])
def test_fork_64_states_into_512_candidates(E, f64):
    import torch
    g, m = 64, 512
    src = _make(E, g, f64=f64, **K5)
    _spread(E, src)
    blob = src.save_state()
    dst = _make(E, g * m, f64=f64, **K5)
    dst.reset()
    k = torch.arange(g * m, dtype=torch.int32, device="cuda")
    dst.load_state(blob, blob_indices=k // m)
    for f in ("h", "Vx", "wz", "deltaz", "tick", "ep_idx", "flags", "last_ret"):
        assert _same(dst.get(f), np.repeat(src.get(f), m)), f
    rng = np.random.default_rng(21)
    a_src = rng.uniform(-1, 1, (T, g)).astype(src.np_dtype)
    a_dst = rng.uniform(-1, 1, (T, g * m)).astype(src.np_dtype)
    a_dst[:, ::m] = a_src
    hs = _outputs(E, src, torch.from_numpy(a_src).cuda())
    hd = _outputs(E, dst, torch.from_numpy(a_dst).cuda())
    assert _until_first_done(hs, np.arange(g), hd, np.arange(g) * m) == g
    src.close()
    dst.close()


def test_full_tier_follows_the_blob(E, tmp_path):
    import torch
    n = 4096
    src = _make(E, n, **K5)
    src.reset()
    eps = [E.episode([0, 11000, 259.1667, 0, 0, 0], vref=0.02, use_ctrl=True)] * n
    src.reset_to(eps)
    acts = torch.from_numpy(np.random.default_rng(2).uniform(-1, 1, (T, n)).astype(np.float32)).cuda()
    _outputs(E, src, acts[:5])
    blob = src.save_state()
    dst, plain = _make(E, n, **K5), _make(E, n, **K5)
    _, obs, rew, done, term = plain.alloc_io(terminal_obs=True)
    ev = _profiled(lambda: (plain.step(acts[0], obs, rew, done, term), plain.synchronize()), tmp_path / "plain.json")
    assert [_template_args(e["name"])[0] for e in ev] == [0]
    dst.load_state(blob)
    ev = _profiled(lambda: (dst.step(acts[0], obs, rew, done, term), dst.synchronize()), tmp_path / "loaded.json")
    assert [_template_args(e["name"])[0] for e in ev] == [3], [e["name"] for e in ev]
    dst.load_state(blob)
    ha, hb = _outputs(E, src, acts), _outputs(E, dst, acts)
    for key in ha:
        assert _same(ha[key], hb[key]), key
    for e in (src, dst, plain):
        e.close()


def _raw(E, eng, blob, blob_idx=None, env_idx=None, n=None):
    """b747_load_state itself: its return code (the index and blob tensors are complete before the call)."""
    import torch
    from b747_rl_ctrl_b200 import _lib
    torch.cuda.synchronize()
    p = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
    n = eng.n_envs if n is None else n
    return _lib.load().b747_load_state(eng._h, p(blob), p(blob_idx), p(env_idx), n)


def test_rejected_blobs_write_nothing(E):
    from b747_rl_ctrl_b200 import _lib
    n = 300
    dst = _make(E, n, **K5)
    _spread(E, dst)
    probe = dst.get("h").copy()
    cases = {"f64 blob": _make(E, n, f64=True, **K5), "obs_type": _make(E, n, obs_type=1, **K5),
             "record_capacity": _make(E, n, record_capacity=5, **K5)}
    for what, other in cases.items():
        other.reset()
        assert _raw(E, dst, other.save_state()) == _lib.ERR_STATE, what
        with pytest.raises(E.B747Error):
            dst.load_state(other.save_state())
        with pytest.raises(E.B747Error):   # the other way round the foreign blob is the smaller one
            other.load_state(dst.save_state())
        other.close()
    same = _make(E, n, seed=99, env_id_offset=500, **K5)   # seed and env ids are not part of the key
    same.reset()
    bad = same.save_state()
    bad[0] ^= 0xFF
    assert _raw(E, dst, bad) == _lib.ERR_STATE
    bad = same.save_state()
    bad[4] += 1   # format version
    assert _raw(E, dst, bad) == _lib.ERR_STATE
    assert _same(dst.get("h"), probe)
    assert _raw(E, dst, same.save_state()) == _lib.OK
    assert _same(dst.get("h"), same.get("h"))
    dst.close()
    same.close()


def test_out_of_range_indices_are_skipped(E):
    import torch
    from b747_rl_ctrl_b200 import _lib
    n = 300
    src, dst = _make(E, n, seed=1, **K5), _make(E, n, seed=2, **K5)
    _spread(E, src)
    dst.reset()
    blob = src.save_state(np.array([3, -1, 7, n, 1 << 30], np.int32))   # entries 1, 3, 4 are skipped
    before = _fields(E, dst)
    env_idx = torch.tensor([10, 11, -5, 12, 13, n, 14], dtype=torch.int32, device="cuda")
    blob_idx = torch.tensor([0, 2, 0, -1, 5, 2, 1 << 30], dtype=torch.int32, device="cuda")
    assert _raw(E, dst, blob, blob_idx, env_idx, 7) == _lib.OK   # only (10 <- 0) and (11 <- 2) are in range
    after, ref = _fields(E, dst), _fields(E, src)
    moved = {10: 3, 11: 7}
    for f in after:
        for i in range(n):
            want = ref[f][moved[i]] if i in moved else before[f][i]
            assert _same(after[f][i:i + 1], np.array([want])), (f, i)
    # n > n_envs with the identity map
    out = torch.empty(src.state_bytes(n + 1), dtype=torch.uint8, device="cuda")
    assert _lib.load().b747_save_state(src._h, None, n + 1, ctypes.c_void_p(out.data_ptr())) == _lib.ERR_ARG
    assert _raw(E, dst, src.save_state(), n=n + 1) == _lib.ERR_ARG
    src.close()
    dst.close()


def test_misaligned_pointers_are_refused(E):
    """Blobs and index arrays off their 16- / 4-byte alignment are B747_ERR_ARG before any launch; the Python layer
    refuses a misaligned `out` and loads a misaligned blob through an aligned copy."""
    import torch
    from b747_rl_ctrl_b200 import _lib
    L = _lib.load()
    n = 300
    src, dst = _make(E, n, seed=1, **K5), _make(E, n, seed=2, **K5)
    _spread(E, src)
    dst.reset()
    probe = dst.get("h").copy()
    blob = src.save_state()
    nb = blob.numel()
    buf = torch.full((nb + 16,), 0xAB, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    for off in (1, 4, 8):
        assert L.b747_save_state(src._h, None, n, ctypes.c_void_p(buf.data_ptr() + off)) == _lib.ERR_ARG, off
    src.synchronize()
    assert bool((buf == 0xAB).all())
    buf[8:8 + nb].copy_(blob)
    assert _raw(E, dst, buf[8:8 + nb]) == _lib.ERR_ARG
    idx = torch.arange(8, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    bad_idx = ctypes.c_void_p(idx.data_ptr() + 2)
    assert L.b747_load_state(dst._h, ctypes.c_void_p(blob.data_ptr()), bad_idx, None, 4) == _lib.ERR_ARG
    assert L.b747_load_state(dst._h, ctypes.c_void_p(blob.data_ptr()), None, bad_idx, 4) == _lib.ERR_ARG
    out = torch.empty(nb + 16, dtype=torch.uint8, device="cuda")
    assert L.b747_save_state(src._h, bad_idx, 4, ctypes.c_void_p(out.data_ptr())) == _lib.ERR_ARG
    assert _same(dst.get("h"), probe)
    with pytest.raises(ValueError):
        src.save_state(out=out[8:])
    dst.load_state(buf[8:8 + nb])
    assert _same(dst.get("h"), src.get("h")) and not _same(probe, src.get("h"))
    src.close()
    dst.close()


def test_python_round_trip(E):
    import torch
    from b747_rl_ctrl_b200.vec_env import B747VecEnv
    n = 1000
    a = _make(E, n, **K5)
    _spread(E, a)
    cpu = a.save_state().cpu()   # what a checkpoint on disk holds
    b = _make(E, n, **K5)
    b.load_state(cpu)
    acts = torch.from_numpy(np.random.default_rng(4).uniform(-1, 1, (T, n)).astype(np.float32)).cuda()
    ha, hb = _outputs(E, a, acts), _outputs(E, b, acts)
    for key in ha:
        assert _same(ha[key], hb[key]), key
    a.close()
    b.close()

    def roll(env, acts):
        out = []
        for k in range(len(acts)):
            obs, rew, done, infos = env.step(acts[k])
            term = [infos[i]["terminal_observation"] for i in np.flatnonzero(done)]
            out.append((obs.copy(), rew.copy(), done.copy(), np.array(term)))
        return out

    v = B747VecEnv(n, tk=1.0, seed=5)
    v.reset()
    acts = np.random.default_rng(6).uniform(-1, 1, (T, n)).astype(np.float32)
    roll(v, acts[:7])
    st = v.get_state()
    first = roll(v, acts)
    obs0 = v.set_state(st)
    assert _same(obs0, st["obs"])
    second = roll(v, acts)
    w = B747VecEnv(n, tk=1.0, seed=5)
    obs1 = w.set_state({**st, "engine": st["engine"].cpu()})
    assert _same(obs1, st["obs"])
    third = roll(w, acts)
    assert sum(int(x[2].sum()) for x in first) >= n
    for k in range(T):
        for j in range(4):
            assert _same(first[k][j], second[k][j]) and _same(first[k][j], third[k][j]), (k, j)
    v.close()
    w.close()
