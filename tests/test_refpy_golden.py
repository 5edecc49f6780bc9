"""The env layer pinned to the reference's OWN Python.

tests/golden/env_golden_refpy.npz (+ env_golden_refpy_2.npz) holds trajectories produced by the reference's
env/ctrl_env.py + core/controller.py + core/model.py themselves (unmodified, imported in place, over the DLL's own machine code; generator:
tests/golden/make_env_golden_refpy.py, provenance line inside the file).  Checked here:
  * the reference's Controller.reset, fed the Philox stream, lands on exactly the episode the oracle's
    b747o_env_draw_episode draws (distributions AND draw order, every family);
  * the oracle's C env layer over the DLL reproduces observation / reward / done BIT FOR BIT;
  * the float64 restatement tracks it within the float64 bar;
  * (GPU) the float64 kernel does, through the C ABI.
"""
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)


def _golden():
    # stored as two files to keep each under 1 MB: the families with a PID in the loop are in the second
    g = {}
    for f in ("env_golden_refpy.npz", "env_golden_refpy_2.npz"):
        g.update(np.load(os.path.join(HERE, "golden", f)))
    meta = json.loads(bytes(g["meta_json"]).decode())
    return g, meta


def _cfg(O, m):
    return O.make_cfg(seed=m["seed"], **m["kw"])


def _explicit(m):
    """Families rolled from explicit episodes (Controller.reset(state0) + constant reference function)."""
    return m["kw"].get("reset_ref_mode", 0) == -1


def _episodes(mod, g, name, m):
    """The explicit episodes of a family as `mod.episode(...)` descriptors (mod = oracle or engine)."""
    rows = g[name + "/episodes"][:, 0]
    return [mod.episode(r[:6], vref=r[7], h_ref=r[8], use_ctrl=bool(r[6]), aero_err=r[16:21]) for r in rows]


def test_provenance_says_reference_python():
    _, meta = _golden()
    assert "/root/reference/env/ctrl_env.py" in meta["provenance"] and "unmodified" in meta["provenance"]
    assert set(meta["families"]) >= {"canonical", "K10", "speed_addproc", "state_angvel_hybrid_dist", "quality_semimanual",
                                     "tfref_unnormalised", "aero_adddirect_osc"}


def test_reset_draws_match_reference_reset_code(oracle):
    """Controller.reset (core/controller.py:134-193) consuming the Philox stream == b747o_env_draw_episode."""
    g, meta = _golden()
    n_checked = 0
    for name, m in meta["families"].items():
        if _explicit(m):
            continue
        cfg = _cfg(oracle, m)
        eps = g[name + "/episodes"]          # [n, E, 21]
        for e in range(m["n"]):
            for k in range(eps.shape[1]):
                ep = oracle.draw_episode(cfg, e, k)
                row = eps[e, k]
                assert list(ep.state0) == list(row[:6]), (name, e, k)
                use_ctrl = bool(row[6])
                assert bool(ep.use_ctrl) == use_ctrl, (name, e, k)
                if use_ctrl:
                    assert ep.h_ref == row[8], (name, e, k)
                elif row[9]:
                    assert ep.oscillating and list(ep.osc_A) == list(row[10:13]) and list(ep.osc_f) == list(row[13:16])
                else:
                    assert ep.vref_const == row[7], (name, e, k)
                assert list(ep.aero_err) == list(row[16:21]), (name, e, k)
                n_checked += 1
    assert n_checked >= 100
    assert {n for n, m in meta["families"].items() if _explicit(m)} == {"auto_none_explicit", "fullauto_none_explicit",
                                                                        "manual_explicit_addproc"}


def test_c_env_layer_over_dll_is_bit_identical_to_reference_python(oracle, dllref):
    g, meta = _golden()
    for name, m in meta["families"].items():
        cfg = _cfg(oracle, m)
        for e in range(m["n"]):
            env = oracle.RefEnv(cfg, env_id=e)
            assert ((env.reset_to(_episodes(oracle, g, name, m)[e]) if _explicit(m) else env.reset()) == 0).all()
            obs, rew, done = env.rollout(g[name + "/actions"][e], auto_reset=True)
            assert np.array_equal(done, g[name + "/done"][e].astype(bool)), (name, e)
            assert np.array_equal(obs, g[name + "/obs"][e]), (name, e, np.abs(obs - g[name + "/obs"][e]).max())
            assert np.array_equal(rew, g[name + "/rew"][e]), (name, e, np.abs(rew - g[name + "/rew"][e]).max())


def _compare(step, g, name, m, obs_tol, rew_tol):
    acts = g[name + "/actions"]
    for k in range(m["steps"]):
        term, rew, done = step(acts[:, k])
        ref = g[name + "/obs"][:, k]
        assert np.array_equal(done.astype(bool), g[name + "/done"][:, k].astype(bool)), (name, k)
        assert (np.abs(term - ref) <= obs_tol[0] + obs_tol[1] * np.abs(ref)).all(), (name, k, np.abs(term - ref).max())
        assert np.abs(rew - g[name + "/rew"][:, k]).max() <= rew_tol, (name, k, np.abs(rew - g[name + "/rew"][:, k]).max())


def test_restatement_tracks_reference_python(oracle):
    g, meta = _golden()
    for name, m in meta["families"].items():
        ob = oracle.OracleBatch(_cfg(oracle, m), m["n"])
        ob.reset_to(_episodes(oracle, g, name, m)) if _explicit(m) else ob.reset()

        def step(a):
            _, r, d, t = ob.step(a)
            return t, r, d
        # the disturbed / altitude-loop families amplify the libm last-bit differences between the restatement and the DLL
        loose = name in ("state_angvel_hybrid_dist", "quality_semimanual")
        _compare(step, g, name, m, (1e-10, 1e-9) if loose else (1e-12, 1e-9), 1e-9)


@pytest.mark.gpu
def test_f64_kernel_tracks_reference_python():
    from b747_rl_ctrl_b200 import engine as E
    g, meta = _golden()
    for name, m in meta["families"].items():
        eng = E.BatchEngine(n_envs=m["n"], dtype=E.F64, seed=m["seed"], auto_reset=True, **m["kw"])
        eng.reset_to(_episodes(E, g, name, m)) if _explicit(m) else eng.reset()
        term = np.zeros((m["n"], eng.obs_dim))

        def step(a):
            nonlocal term
            _, r, d, term = eng.step_host(a, terminal_obs=term)
            return term, r, d
        loose = name in ("state_angvel_hybrid_dist", "quality_semimanual")
        _compare(step, g, name, m, (1e-10, 1e-9) if loose else (1e-12, 1e-9), 1e-9)
        eng.close()


@pytest.mark.gpu
def test_f32_kernel_tracks_reference_python():
    """The throughput path against the reference's own Python: the per-family bounds of test_gpu_parity (these
    trajectories stay inside the flight envelope)."""
    from b747_rl_ctrl_b200 import engine as E
    from test_gpu_parity import FAMILY_BOUNDS
    g, meta = _golden()
    for name, m in meta["families"].items():
        ob, rb, _ = FAMILY_BOUNDS.get(name, (1e-6, 2e-3, 0.0))
        eng = E.BatchEngine(n_envs=m["n"], dtype=E.F32, seed=m["seed"], auto_reset=True, **m["kw"])
        eng.reset_to(_episodes(E, g, name, m)) if _explicit(m) else eng.reset()
        term = np.zeros((m["n"], eng.obs_dim), np.float32)
        acts = g[name + "/actions"]
        for k in range(m["steps"]):
            _, r, d, term = eng.step_host(acts[:, k].astype(np.float32), terminal_obs=term)
            ref = g[name + "/obs"][:, k]
            assert np.array_equal(d.astype(bool), g[name + "/done"][:, k].astype(bool)), (name, k)
            assert (np.abs(term - ref) <= ob * (1 + np.abs(ref))).all(), (name, k, np.abs(term - ref).max())
            assert np.abs(r - g[name + "/rew"][:, k]).max() <= rb + 0.08, (name, k)
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["manual_explicit_addproc", "auto_none_explicit", "fullauto_none_explicit"])
def test_gym_facade_replays_reference_python(name):
    """The single-env ControllerEnv / Controller facade (gym 0.19 API) driven exactly like the reference's env in the
    golden generator -- constructor with constant reference functions, reset(state0), step, reset() on done -- returns the
    reference's observations, rewards and done flags."""
    from b747_rl_ctrl_b200.core.controller import CtrlMode, CtrlType
    from b747_rl_ctrl_b200.env.ctrl_env import ControllerEnv, ObservationType, RewardType
    g, meta = _golden()
    m = meta["families"][name]
    kw = m["kw"]
    for e in range(2):
        row = g[name + "/episodes"][e, 0]
        env = ControllerEnv(ObservationType(kw.get("obs_type", 0)), RewardType(kw.get("rew_type", 0)), True, True,
                            CtrlType(kw.get("ctrl_type", 3)), None if kw.get("ctrl_mode", 0) < 0 else CtrlMode(kw["ctrl_mode"]),
                            vartheta_func=lambda _, v=row[7]: v, h_func=lambda _, h=row[8]: h, reset_ref_mode=None,
                            tk=kw.get("tk", 20.0), sample_time=0.05, action_max=kw.get("action_max", 17 * np.pi / 180))
        obs = env.reset(np.array(row[:6]))
        assert (obs == 0).all()
        n_done = 0
        for k in range(200):
            a = np.array([g[name + "/actions"][e, k]])
            obs, r, done, info = env.step(a)
            ref = g[name + "/obs"][e, k]
            assert done == bool(g[name + "/done"][e, k]) and info == {}, (name, e, k)
            assert np.allclose(obs, ref, rtol=1e-9, atol=1e-12), (name, e, k, np.abs(obs - ref).max())
            assert abs(r - g[name + "/rew"][e, k]) <= 1e-9, (name, e, k)
            if done:
                n_done += 1
                env.reset()
        assert n_done == 2
        env.close()
