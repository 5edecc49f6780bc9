#!/usr/bin/env python
"""Golden trajectories of the ENV LAYER produced by the reference's own Python -- /root/reference/env/ctrl_env.py,
core/controller.py and core/model.py, unmodified, imported from where they lie -- on top of the reference DLL's own
machine code (oracle/refpy.py, oracle/_ref/model_simple.so).  Needs /root/reference: run in the build container;
the output tests/golden/env_golden_refpy.npz + env_golden_refpy_2.npz is committed; the tests read only that.

For every configuration family of the parity tests, N envs are rolled through more than one episode the way a
SubprocVecEnv worker does it (`obs, r, done, info = env.step(a)`; on done `env.reset()`), with float64 actions that
are exactly representable in float32.  Controller.reset's random draws come from the Philox stream of the oracle /
CUDA path (refpy.PhiloxRandom behind the module's `random` and `np.random`), consumed by the REFERENCE's reset code in
its own order; the episode it lands on is recorded next to the trajectory.

  <family>/actions [N, T]  <family>/obs [N, T, O]  <family>/rew [N, T]  <family>/done [N, T]
  <family>/episodes [N, E, 21]: state0[6], use_ctrl, vref, href, oscillating, A[3], f[3], aero_err[5] of every reset
"""
import json
import math
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import refpy  # noqa: E402

DEG = math.pi / 180
SEED = 9
# the families of tests/test_gpu_parity.py VARIANTS (kwargs of engine.make_cfg / oracle.make_cfg) + the canonical one
FAMILIES = {
    "canonical": dict(),
    "K10": dict(sample_time=0.10),
    "K1_tk3": dict(sample_time=None, tk=3.0),
    "speed_addproc": dict(obs_type=1, ctrl_mode=1, action_max=1.0),
    "aero_adddirect_osc": dict(obs_type=3, ctrl_mode=3, action_max=10 * DEG, reset_ref_mode=1),
    "state_angvel_hybrid_dist": dict(obs_type=4, ctrl_mode=2, action_max=2 * DEG, reset_ref_mode=2, disturbance_mode=0),
    "pidaero_pidlike_limiter": dict(obs_type=2, rew_type=1, use_limiter=True),
    "quality_semimanual": dict(rew_type=2, ctrl_type=2, reset_ref_mode=2),
    "minimal": dict(rew_type=3),
    "tfref_unnormalised": dict(rew_type=4, norm_obs=False, norm_act=False),
    "fixed_aero_err": dict(disturbance_mode=0, aero_err=[-0.1, 0.1, -0.1, -0.1, 0.1]),
    # explicit episodes (Controller.reset(state0) with a constant reference function, reset_ref_mode None), the СС PID in
    # the loop and ctrl_mode None: the env ControllerAgent.test builds for its PID baseline (neural/agent.py:298-307)
    "auto_none_explicit": dict(ctrl_type=1, ctrl_mode=-1, reset_ref_mode=-1, tk=4.0),
    "fullauto_none_explicit": dict(ctrl_type=0, ctrl_mode=-1, reset_ref_mode=-1, tk=4.0, rew_type=2),
    "manual_explicit_addproc": dict(ctrl_mode=1, action_max=1.0, reset_ref_mode=-1, tk=4.0),
}


def explicit_episode(name, e):
    """(state0, vref, href) of env e of an explicit-episode family."""
    s0 = [0.0, 9000.0 + 500.0 * e, 230.0 + 5.0 * e, float(e - 1), 0.0, 0.0]
    vref = (3.0 + e) * DEG * (-1.0) ** e
    href = s0[1] + 300.0 * (-1.0) ** e
    return s0, vref, href
DEFAULTS = dict(obs_type=0, rew_type=0, ctrl_type=3, ctrl_mode=0, reset_ref_mode=0, disturbance_mode=-1, norm_obs=True,
                norm_act=True, use_limiter=False, tk=20.0, sample_time=0.05, action_max=17 * DEG, vartheta_max=10 * DEG,
                aero_err=None)


def make_ref_env(ref, kw, rng):
    CE, C = ref.ctrl_env, ref.controller
    k = dict(DEFAULTS, **kw)
    refpy.patch_rng(ref, rng)
    env = CE.ControllerEnv(
        CE.ObservationType(k["obs_type"]), CE.RewardType(k["rew_type"]), k["norm_obs"], k["norm_act"],
        C.CtrlType(k["ctrl_type"]), None if k["ctrl_mode"] < 0 else C.CtrlMode(k["ctrl_mode"]),
        vartheta_func=k.get("vartheta_func"), h_func=k.get("h_func"),
        reset_ref_mode=None if k["reset_ref_mode"] < 0 else C.ResetRefMode(k["reset_ref_mode"]),
        disturbance_mode=None if k["disturbance_mode"] < 0 else C.DisturbanceMode(k["disturbance_mode"]),
        tk=k["tk"], sample_time=k["sample_time"], action_max=k["action_max"], vartheta_max=k["vartheta_max"],
        use_limiter=k["use_limiter"], aero_err=None if k["aero_err"] is None else np.array(k["aero_err"], dtype=float))
    return env


def episode_row(ctrl):
    s0, use_ctrl, vref, href, osc, aero = refpy.episode_of(ctrl)
    A, f = osc if osc else ([0, 0, 0], [0, 0, 0])
    return np.array(list(s0) + [float(use_ctrl), vref, href, float(osc is not None)] + list(A) + list(f) + list(aero))


def main():
    ref = refpy.load()
    C = ref.controller
    # every Controller.reset starts a new episode of the Philox stream (the constructor's own reset is episode 0)
    orig_reset = C.Controller.reset
    state = {"rng": None, "rows": None}

    def reset(self, state0=None):
        state["rng"].begin_episode()
        r = orig_reset(self, state0)
        state["rows"].append(episode_row(self))
        return r
    C.Controller.reset = reset
    out, meta = {}, {}
    for name, kw in FAMILIES.items():
        n = 8 if kw.get("reset_ref_mode") == 2 else 4
        steps = 320 if name == "K1_tk3" else 420
        amax = 1.0 if kw.get("norm_act", True) else kw.get("action_max", 17 * DEG)
        arng = np.random.default_rng(SEED)
        acts = arng.uniform(-amax, amax, (steps, n)).astype(np.float32).astype(np.float64).T.copy()   # [n, steps]
        obs = rew = done = None
        eps = []
        for e in range(n):
            rng = refpy.PhiloxRandom(SEED, e)
            rng.episode = -1
            state["rng"], state["rows"] = rng, []
            if kw.get("reset_ref_mode", 0) < 0:    # explicit episode: constant reference functions + reset(state0)
                s0, vref, href = explicit_episode(name, e)
                env = make_ref_env(ref, dict(kw, vartheta_func=lambda _, v=vref: v, h_func=lambda _, h=href: h), rng)
                state["rows"] = []
                env.reset(np.array(s0))
            else:
                env = make_ref_env(ref, kw, rng)   # __init__ resets once: episode 0
            od = env.observation_space.shape[0]
            if obs is None:
                obs, rew, done = np.zeros((n, steps, od)), np.zeros((n, steps)), np.zeros((n, steps), np.uint8)
            for k in range(steps):
                o, r, d, _ = env.step(np.array([acts[e, k]]))
                obs[e, k], rew[e, k], done[e, k] = o, r, d
                if d:
                    env.reset()
            eps.append(np.stack(state["rows"]))
        n_eps = min(len(x) for x in eps)
        out[name + "/actions"], out[name + "/obs"], out[name + "/rew"], out[name + "/done"] = acts, obs, rew, done
        out[name + "/episodes"] = np.stack([x[:n_eps] for x in eps])
        meta[name] = {"kw": {k: (v if not isinstance(v, np.ndarray) else v.tolist()) for k, v in kw.items()}, "n": n,
                      "steps": steps, "seed": SEED, "episodes": int(done.sum())}
        print(f"{name}: {n} envs x {steps} steps, {int(done.sum())} episodes finished, obs dim {obs.shape[2]}, "
              f"return of env 0 {rew[0].sum():.6f}", flush=True)
    out["meta_json"] = np.frombuffer(json.dumps({
        "families": meta,
        "provenance": "obs / reward / done produced by /root/reference/env/ctrl_env.py + core/controller.py + core/model.py "
                      "(unmodified, imported in place) over core/model_simple_win64.dll's own machine code "
                      "(oracle/_ref/model_simple.so); Controller.reset's random/np.random replaced by the Philox stream"}).encode(),
        dtype=np.uint8)
    # the families with a PID in the loop (ctrl_type other than MANUAL) go to a second file, so that neither exceeds 1 MB
    second = {n for n, kw in FAMILIES.items() if kw.get("ctrl_type", 3) != 3}
    np.savez_compressed(os.path.join(HERE, "env_golden_refpy.npz"),
                        **{k: v for k, v in out.items() if k.split("/")[0] not in second})
    np.savez_compressed(os.path.join(HERE, "env_golden_refpy_2.npz"),
                        **{k: v for k, v in out.items() if k.split("/")[0] in second})


if __name__ == "__main__":
    main()
