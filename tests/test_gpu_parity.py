"""GPU parity tests: the CUDA path (through the C ABI) against the oracle on identical seeded
inputs, against the committed DLL golden vectors, and -- at BASELINE.json's full size -- through
size-independent properties.  Bars: float64 mode obs/reward within 1e-9 (relative, with an absolute
floor for the finite-difference signals), done flags / step counts / episode counts bit-exact;
f32 mode within the bound stated in DESIGN.md over 1000-step trajectories, done flags bit-exact."""
import json
import math
import os
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
DEG = math.pi / 180


@pytest.fixture(scope="module")
def E():
    import torch
    assert torch.cuda.is_available()
    from b747_rl_ctrl_b200 import engine
    return engine



# ---- per-step state / signal parity (float64 handles with export_signals) -------------------------------------------
# b747 field name -> (oracle name, index, floor).  The bar is |d| <= 1e-9 * (|ref| + floor): 1e-9 relative (north_star)
# with an absolute floor at the field's resolution of interest, so that zero crossings do not make the bar vacuous.
X_FIELDS = {
    "x": ("X", 0, 1.0), "h": ("X", 1, 1.0), "q0": ("X", 2, 1.0), "q3": ("X", 5, 1e-2), "Vx": ("X", 6, 1.0),
    "Vy": ("X", 7, 1.0), "wz": ("X", 8, 1e-3), "cs_int": ("X", 9, 1e-3), "cs_flt": ("X", 10, 1e-3),
    "ss_int": ("X", 11, 1e-3), "ss_flt": ("X", 12, 1e-3), "dv_int": ("X", 13, 1e-3), "itae": ("X", 14, 1e-3),
    "iae": ("X", 15, 1e-3), "ise": ("X", 16, 1e-4), "itse": ("X", 17, 1e-4),
}
SIG_FIELDS = {
    "sig_state_x": ("state", 0, 1.0), "sig_state_y": ("state", 1, 1.0), "sig_state_Vx": ("state", 2, 1.0),
    "sig_state_Vy": ("state", 3, 1.0), "sig_state_vartheta": ("state", 4, 1e-3), "sig_state_wz": ("state", 5, 1e-3),
    "sig_sim_time": ("sim_time", 0, 0.0), "sig_vartheta_zh": ("vartheta_zh", 0, 1e-3),
    "sig_U_com_PID": ("U_com_PID", 0, 1e-3), "sig_CXa": ("CXa", 0, 1e-3), "sig_CYa": ("CYa", 0, 1e-2),
    "sig_mz": ("mz", 0, 1e-3), "sig_K_alpha": ("K_alpha", 0, 1e-2), "sig_dCm_ddeltaz": ("dCm_ddeltaz", 0, 1e-4),
    "sig_U_com": ("U_com", 0, 1e-3), "sig_deltaz_RP": ("deltaz_RP", 0, 1e-3), "sig_dvartheta": ("dvartheta", 0, 1e-3),
    "sig_dvartheta_int": ("dvartheta_int", 0, 1e-3), "sig_dvartheta_dt": ("dvartheta_dt", 0, 1e-3),
    "sig_TAE": ("TAE", 0, 1e-3), "sig_ITAE": ("ITAE", 0, 1e-3), "sig_TSE": ("TSE", 0, 1e-4),
    "sig_ITSE": ("ITSE", 0, 1e-4), "sig_AE": ("AE", 0, 1e-3), "sig_IAE": ("IAE", 0, 1e-3), "sig_SE": ("SE", 0, 1e-4),
    "sig_ISE": ("ISE", 0, 1e-4), "sig_alpha": ("alpha", 0, 1e-3), "sig_V": ("V", 0, 1.0), "sig_Mach": ("Mach", 0, 1e-2),
}
# the second finite difference over 10 ms amplifies 1-ulp libm differences by 1/h^2 (SURVEY.md 7 hard part 3)
DDT2 = ("sig_dvartheta_dt_dt", "dvartheta_dt_dt", 1e-9, 1e-6)


# Flight envelope (decided from the float64 ORACLE's own signals, never from the output under test): an env is inside
# from its reset until the oracle's angle of attack first leaves |alpha| <= 26 deg or its pitch |theta| <= 80 deg.  26 deg
# is the end of the tabulated aerodynamics (CYa to 25 deg, mz to 17.7 deg, K_alpha's knee at 25-30 deg): beyond it the
# coefficients are linear extrapolations, the airframe tumbles and the motion is chaotic -- any last-bit difference, also
# between the DLL and its float64 restatement, grows without bound; beyond 80 deg of pitch the trajectory runs into the
# DLL's asin(sin theta) fold at +-90 deg.  An env outside is excused until its next reset; tests count the excused
# env-steps and cap their share.
ALPHA_ENV = 0.45
THETA_ENV = 1.40


def _envelope_update(ob, out, d_o):
    """Latch `out` for envs whose oracle state left the envelope in this step (envs that just finished were reset by
    ob.step: their signals are zero and the new episode starts inside)."""
    out |= ((np.abs(ob.gather("alpha")) > ALPHA_ENV) | (np.abs(ob.gather("state", 4)) > THETA_ENV)) & ~d_o
    return ~out


def _field_ratios(eng, ob, ratios, ddt_scale=1.0, inside=None):
    """max over envs of |engine field - oracle field| / bar, accumulated per field into `ratios`.
    ddt_scale widens the floors of the two finite-difference signals (families with unstable members, see
    test_f64_variants_match_oracle)."""
    for name, (oname, idx, floor) in {**X_FIELDS, **SIG_FIELDS}.items():
        ref = ob.gather(oname, idx)
        if name == "sig_dvartheta_dt":
            floor *= ddt_scale
        bar = 1e-9 * (np.abs(ref) + floor)
        bar[bar == 0] = 1e-300   # sim_time: exact
        q = np.abs(eng.get(name) - ref) / bar
        ratios[name] = max(ratios.get(name, 0.0), float((q if inside is None else q[inside]).max(initial=0.0)))
    name, oname, a, r = DDT2
    ref = ob.gather(oname)
    q = np.abs(eng.get(name) - ref) / (ddt_scale * (a + r * np.abs(ref)))
    ratios[name] = max(ratios.get(name, 0.0), float((q if inside is None else q[inside]).max(initial=0.0)))
    assert np.array_equal(eng.get("tick").astype(np.int64), ob.ticks()), "model tick counters differ"


# ---- tunables away from their defaults --------------------------------------------------------------------------------
# Airframe parameters and PID gains are settable per handle (b747_set_param) and, all but g, per env
# (b747_set_env_param / b747_set_env_param_range).  A kernel that read a default instead of the tunable at one site would
# agree with the oracle at the defaults, so the families below also run at these values.
TUNABLES = ("m0", "Iz", "P", "S", "c_", "g", "PID_SS", "PID_CS")
ROW0 = {"m0": 0, "Iz": 1, "P": 2, "S": 3, "c_": 4, "PID_SS": 5, "PID_CS": 9}   # per-env rows, include/b747.h
# batch-wide values: multipliers of the defaults
TUNED_SCALE = {"m0": 1.15, "Iz": 0.9, "P": 1.08, "S": 0.97, "c_": 1.03, "g": 0.998, "PID_SS": [1.2, 0.8, 1.1, 0.9],
               "PID_CS": [0.8, 1.25, 0.9, 1.1]}
# per-env ranges: default x (1 -+ f), every PID component ordered for its sign
RANGE_FRAC = {"m0": 0.2, "Iz": 0.2, "P": 0.1, "S": 0.1, "c_": 0.1, "PID_SS": 0.3, "PID_CS": 0.3}


def tunable_defaults(O):
    """The DLL defaults, as the oracle's model holds them."""
    m = O.CModel()
    return {nm: np.atleast_1d(np.asarray(m.get(nm), np.float64)) for nm in TUNABLES}


def tuned_params(O):
    d = tunable_defaults(O)
    return {nm: d[nm] * np.asarray(TUNED_SCALE[nm]) for nm in TUNABLES}


def tuned_ranges(O):
    d = tunable_defaults(O)
    out = {}
    for nm, f in RANGE_FRAC.items():
        a, b = d[nm] * (1 - f), d[nm] * (1 + f)
        out[nm] = (np.minimum(a, b), np.maximum(a, b))
    return out


class OracleTunables:
    """The tunables of every env of an OracleBatch, kept as the handle under test keeps its own: whole-batch values
    (set_param), per-env values (set_env_param) and ranges drawn at every random reset by the formula of include/b747.h,
    lo + (hi - lo) u with u = the oracle's b747o_uniform53(seed, env id, episode, 32 + row).  The episode index of each
    env is counted from the ORACLE's done flags, so no input of the oracle is read back from the handle under test."""

    def __init__(self, O, ob, cfg_o, env_id_offset=0, reapply_hybrid=True):
        self._L, self.ob, self.seed = O.olib(), ob, cfg_o.seed
        self.hybrid = cfg_o.reset_ref_mode == O.RESET_HYBRID
        self.reapply_hybrid = reapply_hybrid
        self.ids = env_id_offset + np.arange(ob.n)
        self.epi = np.zeros(ob.n, np.int64)
        self.vals = {nm: np.tile(v, (ob.n, 1)) for nm, v in tunable_defaults(O).items()}
        self.ranges = {}

    def set_param(self, name, v):
        """b747_set_param: the batch value, and in per-env mode every env's value of that name."""
        self.vals[name] = np.tile(np.atleast_1d(np.asarray(v, np.float64)), (self.ob.n, 1))
        self._give(range(self.ob.n), [name])

    def set_env_param(self, name, v):
        self.vals[name] = np.asarray(v, np.float64).reshape(self.ob.n, -1).copy()
        self._give(range(self.ob.n), [name])

    def set_range(self, name, lo, hi):
        self.ranges[name] = tuple(np.atleast_1d(np.asarray(x, np.float64)) for x in (lo, hi))

    def _give(self, envs, names=None):
        for i in envs:
            m = self.ob.model(int(i))
            for nm in names if names is not None else self.vals:
                v = self.vals[nm][i]
                m.set(nm, v if len(v) > 1 else v[0])

    def reset(self):
        """After ob.reset(): episode 0 of every env."""
        self.epi[:] = 0
        self._on_reset(np.arange(self.ob.n))

    def step(self, d_o):
        """After ob.step(): the envs that finished started their next episode."""
        envs = np.nonzero(d_o)[0]
        self.epi[envs] += 1
        self._on_reset(envs)

    def _on_reset(self, envs):
        for nm, (lo, hi) in self.ranges.items():
            for i in envs:
                for j in range(len(lo)):
                    u = self._L.b747o_uniform53(self.seed, int(self.ids[i]), int(self.epi[i]), 32 + ROW0[nm] + j)
                    self.vals[nm][i, j] = lo[j] + (hi[j] - lo[j]) * u
        if self.ranges:
            self._give(envs, list(self.ranges))
        if self.hybrid and self.reapply_hybrid:
            reapply_after_hybrid_reset(self, envs)

    def check_handle(self, eng, envs=None):
        """get_env_param of the handle equals the values the oracle flies, bit for bit."""
        envs = np.arange(self.ob.n) if envs is None else np.asarray(envs)
        for nm in self.ranges:
            got = eng.get_env_param(nm).cpu().numpy().reshape(self.ob.n, -1)[envs]
            want = self.vals[nm][envs]
            assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), \
                f"{nm}: handle values differ from lo + (hi - lo) u of the oracle's draw"


def reapply_after_hybrid_reset(tun, envs):
    """A HYBRID reset of the reference re-creates its Model (Controller._init_model; oracle/b747_env_ref.c), which puts
    PID_SS, PID_CS, P and the use_* switches back to the DLL defaults.  The kernels keep the handle's and every env's
    tunables across every reset: they are configuration (include/b747.h at b747_set_param, DESIGN.md section 7).  So
    the oracle is given the handle's values again after each of its HYBRID resets."""
    tun._give(envs)


def _with_tunables(O, eng, ob, cfg_o, params=None, ranges=None, reapply_hybrid=True):
    """Apply batch-wide `params` and per-env `ranges` to the handle and build the oracle's side of them."""
    tun = OracleTunables(O, ob, cfg_o, reapply_hybrid=reapply_hybrid)
    for nm, v in (params or {}).items():
        eng.set_param(nm, v)
        tun.set_param(nm, v)
    for nm, (lo, hi) in (ranges or {}).items():
        eng.set_env_param_range(nm, lo, hi)
        tun.set_range(nm, lo, hi)
    return tun


def _rollout_compare(E, O, dtype, n, steps, kw, seed, obs_tol, rew_tol, sticky=0, fields=False, ddt_scale=1.0,
                     max_excused=0.02, params=None, ranges=None, at_step=None, reapply_hybrid=True, ekw=None):
    """Step engine and oracle in lock-step with the same actions; every env is held to the tolerance at every step
    inside the flight envelope (max_excused: largest share of env-steps outside it).  Done flags,
    step counts and tick counters are compared for all envs.  Returns the worst deviations.
    params: batch-wide tunables, ranges: per-env ranges, both given to the handle and to every oracle env;
    at_step: {k: fn(eng, tun)} called before step k; ekw: engine-only keywords."""
    cfg_o = O.make_cfg(seed=seed, **kw)
    eng = E.BatchEngine(n_envs=n, dtype=dtype, seed=seed, auto_reset=True, **{"export_signals": fields, **(ekw or {})},
                        **kw)
    ob = O.OracleBatch(cfg_o, n)
    tun = _with_tunables(O, eng, ob, cfg_o, params, ranges, reapply_hybrid)
    ratios = {}
    eng.reset()
    o0 = ob.reset()
    tun.reset()
    tun.check_handle(eng)
    assert (o0 == 0).all()
    rng = np.random.default_rng(seed)
    amax = 1.0 if cfg_o.norm_act else cfg_o.action_max
    worst_o = worst_r = 0.0
    env_worst = np.zeros(n)
    term = np.zeros((n, eng.obs_dim), eng.np_dtype)
    n_done = excused = 0
    out = np.zeros(n, bool)
    for k in range(steps):
        if sticky and k % sticky:
            pass  # hold the previous action: drives the airframe far out of the trimmed envelope
        else:
            a = rng.uniform(-amax, amax, n).astype(eng.np_dtype)
        if at_step and k in at_step:
            at_step[k](eng, tun)
        obs, rew, done, term = eng.step_host(a, terminal_obs=term)
        o_o, r_o, d_o, t_o = ob.step(a.astype(np.float64))
        assert np.array_equal(done.astype(bool), d_o), f"done flags differ at step {k}"
        n_done += int(d_o.sum())
        if d_o.any():
            tun.step(d_o)
            tun.check_handle(eng, np.nonzero(d_o)[0])
        ins = _envelope_update(ob, out, d_o)
        excused += int(out.sum())
        eo = np.abs(obs.astype(np.float64) - o_o)[ins]
        et = np.abs(term.astype(np.float64) - t_o)[ins]
        er = np.abs(rew.astype(np.float64) - r_o)[ins]
        lim = obs_tol[0] + obs_tol[1] * np.abs(t_o[ins])
        assert (et <= lim).all(), f"step {k}: terminal/obs deviation {et.max():.3e}"
        assert (eo <= obs_tol[0] + obs_tol[1] * np.abs(o_o[ins])).all(), f"step {k}: obs deviation {eo.max():.3e}"
        assert (er <= rew_tol).all(), f"step {k}: reward deviation {er.max():.3e}"
        worst_o, worst_r = max(worst_o, et.max(initial=0.0)), max(worst_r, er.max(initial=0.0))
        env_worst[ins] = np.maximum(env_worst[ins], et.max(axis=1))
        if fields:
            _field_ratios(eng, ob, ratios, ddt_scale, ins)
        out &= ~d_o
    assert excused <= max_excused * n * steps, f"{excused} of {n * steps} env-steps outside the flight envelope"
    if fields:
        bad = {k: v for k, v in ratios.items() if not v <= 1.0}
        print("state/signal deviation / bar, worst fields:", sorted(ratios.items(), key=lambda kv: -kv[1])[:6])
        assert not bad, f"fields outside 1e-9 relative (deviation / bar): {bad}"
    st = eng.episode_stats()
    assert st[0] == n_done
    eng.env_worst = env_worst
    return worst_o, worst_r, n_done, eng


# ---- fp32 mode: the stated bounds, asserted on EVERY env at EVERY step ------------------------------------------------
# The f32 path is a float32 re-formulation of a HYBRID system (saturations, a clamping anti-windup with a Memory block, a
# rate limiter, a 20 Hz zero-order hold, reward branches).  Two things are therefore part of the statement, and both are
# decided from the float64 ORACLE's own signals, never from the f32 output:
#  * flight envelope (ALPHA_ENV / THETA_ENV above): the bound is stated for an env from its reset until it first leaves
#    the envelope; the test counts the excused env-steps and caps their share.
#  * reward branch.  The CLASSIC reward jumps by up to 0.2 (1 - exp(-kt t)) <= 0.072 where |dvartheta / vf| crosses 0.05
#    (r3, env/ctrl_env.py:133-136); an env whose oracle value sits within REW_EDGE of that threshold may take the other
#    branch, so its reward bar is widened by that jump for that step.
REW_EDGE = 2e-3
REW_JUMP = 0.08


def _reward_edge(O, cfg_o, ob, t_o, d_o):
    """Envs whose oracle pitch error sits within REW_EDGE of the CLASSIC reward's r3 threshold in this step (and envs
    that were just reset, whose reference is gone); all False for the other reward types."""
    edge = np.zeros(len(d_o), bool)
    if cfg_o.rew_type == O.REW_CLASSIC and cfg_o.obs_type != O.OBS_MODEL_STATE:
        dv = t_o[:, 1] * (math.pi if cfg_o.norm_obs else 1.0)
        vr = np.where(ob.gather("use_PID_CS") >= 1.0, ob.gather("vartheta_zh"), ob.gather("vartheta"))
        vr = np.where(d_o, np.nan, vr)   # reset envs: the reference of the finished episode is gone
        vf = np.where(vr != 0, vr, cfg_o.vartheta_max)
        edge = np.abs(np.abs(dv / vf) - 0.05) <= REW_EDGE
        edge |= np.isnan(vr)
    return edge


def _f32_bound_rollout(E, O, n, steps, kw, seed, sticky=0, ekw=None, params=None, ranges=None, at_step=None):
    """f32 engine against the oracle; returns per-step worst deviations inside the envelope and the bookkeeping the
    bound tests assert on.  Done flags are compared bit for bit for ALL envs, excused or not.  ekw: engine-only
    keywords; params, ranges, at_step: as in _rollout_compare."""
    cfg_o = O.make_cfg(seed=seed, **kw)
    eng = E.BatchEngine(n_envs=n, dtype=E.F32, seed=seed, auto_reset=True, **kw, **(ekw or {}))
    ob = O.OracleBatch(cfg_o, n)
    tun = _with_tunables(O, eng, ob, cfg_o, params, ranges)
    eng.reset()
    ob.reset()
    tun.reset()
    tun.check_handle(eng)
    rng = np.random.default_rng(seed)
    amax = 1.0 if cfg_o.norm_act else cfg_o.action_max
    out = np.zeros(n, bool)                      # env left the envelope in its running episode
    res = dict(obs=np.zeros(n), rew=np.zeros(n), rew_edge=np.zeros(n), obs_all=np.zeros(n), excused=0, total=0, n_done=0,
               edge_steps=0)
    term = np.zeros((n, eng.obs_dim), np.float32)
    for k in range(steps):
        if not (sticky and k % sticky):
            a = rng.uniform(-amax, amax, n).astype(np.float32)
        if at_step and k in at_step:
            at_step[k](eng, tun)
        obs, rew, done, term = eng.step_host(a, terminal_obs=term)
        o_o, r_o, d_o, t_o = ob.step(a.astype(np.float64))
        assert np.array_equal(done.astype(bool), d_o), f"done flags differ at step {k}"
        assert np.isfinite(obs).all() and np.isfinite(rew).all()
        if d_o.any():
            tun.step(d_o)
            tun.check_handle(eng, np.nonzero(d_o)[0])
        res["n_done"] += int(d_o.sum())
        inside = _envelope_update(ob, out, d_o)
        eo = (np.abs(term.astype(np.float64) - t_o) / (1.0 + np.abs(t_o))).max(axis=1)   # relative to 1 + |obs|
        er = np.abs(rew.astype(np.float64) - r_o)
        edge = _reward_edge(O, cfg_o, ob, t_o, d_o)
        res["obs_all"] = np.maximum(res["obs_all"], eo)
        res["obs"] = np.maximum(res["obs"], np.where(inside, eo, 0.0))
        res["rew"] = np.maximum(res["rew"], np.where(inside & ~edge, er, 0.0))
        res["rew_edge"] = np.maximum(res["rew_edge"], np.where(inside & edge, er, 0.0))
        res["excused"] += int(out.sum())
        res["edge_steps"] += int((inside & edge).sum())
        res["total"] += n
        out &= ~d_o                              # a reset starts a new episode inside the envelope
    st = eng.episode_stats()
    assert st[0] == res["n_done"]
    eng.close()
    return res


def _assert_bound(name, res, obs_bound, rew_bound, max_excused):
    q = np.quantile(res["obs"], [0.5, 0.99])
    msg = (f"f32 {name}: per-env worst |d obs|/(1+|obs|) median {q[0]:.1e} p99 {q[1]:.1e} max {res['obs'].max():.2e} "
           f"(bound {obs_bound:.0e}); |d rew| max {res['rew'].max():.2e} (bound {rew_bound:.0e}), at a reward branch edge "
           f"{res['rew_edge'].max():.2e} over {res['edge_steps']} env-steps; outside the envelope {res['excused']} of "
           f"{res['total']} env-steps; episodes {res['n_done']}")
    print(msg)
    assert res["obs"].max() <= obs_bound, msg
    assert res["rew"].max() <= rew_bound, msg
    assert res["rew_edge"].max() <= rew_bound + REW_JUMP, msg
    assert res["excused"] <= max_excused * res["total"], msg


# float64 bars.  Observations: 1e-9 relative with a floor of 1e-12 (normalised units; measured <= 7e-14 -- the old 2e-9 floor
# was 1e-4 relative on dvartheta_int / 60 pi early in an episode); rewards 1e-10 (measured 2e-12: the CLASSIC reward reads
# dvartheta_dt_dt, the 1/h^2-amplified signal, through exp(-0.4 |.| / |vref|)).
F64_OBS_TOL = (1e-12, 1e-9)
F64_REW_TOL = 1e-10


def test_f64_matches_oracle_config2(E, oracle):
    """BASELINE configs[1]: 4096 envs x 1000 env steps, float64, per-step parity of observation / reward / done AND of
    the model itself: the 16 continuous states, every exported signal (stage-4 values) and the tick counter of every
    env after every env step, within 1e-9 relative (dvartheta_dt_dt: 1e-9 + 1e-6 relative, SURVEY.md 7.3)."""
    wo, wr, nd, _ = _rollout_compare(E, oracle, E.F64, 4096, 1000, dict(), 5, F64_OBS_TOL, F64_REW_TOL, fields=True)
    assert nd == 4096 * 2  # two auto-resets per env in 1000 steps of 400-step episodes
    print(f"f64 4096x1000: max|dobs|={wo:.2e} max|drew|={wr:.2e}")


VARIANTS = {
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
}


# Families run with every airframe parameter and PID gain away from its default (tuned_params: set_param on the handle and
# on every oracle env): name -> (family of VARIANTS or "canonical", engine-only keywords).
TUNED = {
    "tuned_canonical": ("canonical", None),
    "tuned_K10": ("K10", None),
    "tuned_K1_tk3": ("K1_tk3", None),
    "tuned_speed_addproc": ("speed_addproc", None),
    "tuned_quality_semimanual": ("quality_semimanual", None),
    "tuned_canonical_full": ("canonical", dict(export_signals=True, track_transfer=True, record_capacity=16)),
}
TUNED_F64 = ["tuned_canonical", "tuned_speed_addproc", "tuned_quality_semimanual"]
TUNED_F32 = ["tuned_K10", "tuned_K1_tk3", "tuned_speed_addproc", "tuned_quality_semimanual", "tuned_canonical_full"]


@pytest.mark.parametrize("name", sorted(VARIANTS) + TUNED_F64)
def test_f64_variants_match_oracle(E, oracle, name):
    fam = TUNED[name][0] if name in TUNED else name
    kw = VARIANTS.get(fam, {})
    params = tuned_params(oracle) if name in TUNED else None
    steps = 320 if fam == "K1_tk3" else 420
    # un-normalised observations carry raw magnitudes (Vx ~ 250): relative bar only
    # Aero disturbance N(-+0.1, 0.5) on the five coefficients makes some members of this family open-loop unstable: a few
    # leave the flight envelope and tumble (excused from there to their next reset, at most 5 % of the env-steps), and the
    # ones that stay inside still amplify ANY last-bit difference (the restatement against the DLL itself diverges to
    # 4e-14 on these envs within one episode, tools/family_probe.py `dll`), which the two finite-difference signals
    # multiply by 1/h = 100 and 1/h^2.  States and every other signal keep the 1e-9 bar; the floors of dvartheta_dt /
    # dvartheta_dt_dt are widened by 1/h for this family only (measured round 2: 6.7x / 19x the canonical floors).
    dist = fam == "state_angvel_hybrid_dist"
    wo, wr, nd, _ = _rollout_compare(E, oracle, E.F64, 512, steps, kw, 9, F64_OBS_TOL, F64_REW_TOL, fields=True,
                                     ddt_scale=100.0 if dist else 1.0, max_excused=0.05 if dist else 0.02,
                                     params=params)
    assert nd >= 512
    print(f"f64 {name}: max|dobs|={wo:.2e} max|drew|={wr:.2e} episodes={nd}")


def test_f64_matches_dll_golden(E):
    """The kernels against trajectories produced by the reference DLL's own machine code."""
    g = np.load(os.path.join(HERE, "golden", "env_golden.npz"))
    meta = json.loads(bytes(g["meta_json"]).decode())
    for name, m in meta.items():
        eng = E.BatchEngine(n_envs=m["n"], dtype=E.F64, seed=m["seed"], auto_reset=True, **m["kw"])
        eng.reset()
        acts = g[name + "/actions"]
        term = np.zeros((m["n"], eng.obs_dim))
        for k in range(m["steps"]):
            obs, rew, done, term = eng.step_host(acts[:, k], terminal_obs=term)
            assert np.array_equal(done, g[name + "/done"][:, k]), (name, k)
            ref = g[name + "/obs"][:, k]
            assert (np.abs(term - ref) <= 2e-9 + 1e-9 * np.abs(ref)).all(), (name, k, np.abs(term - ref).max())
            assert np.abs(rew - g[name + "/rew"][:, k]).max() <= 1e-9, (name, k)


def test_f32_bound_over_1000_steps(E, oracle):
    """fp32 mode, canonical config, 1000-step trajectories (2.5 / 5 episodes) of 4096 envs, K = 5 and K = 10.
    Stated bound (DESIGN.md 4.2, README): |d obs| <= 1e-6 (normalised units) and |d reward| <= 2e-3 for EVERY env at EVERY
    step inside the flight envelope, done flags bit-exact for all (measured round 2: 1.2e-7 / 1.6e-7 at K = 5 / 10, p99
    1.1e-7; rewards 4e-4 / 1.2e-3).  Round 1's 1e-5 with excursions to 2.5e-5 came from envs tumbling through the pitch
    fold at theta = +-90 deg -- outside the envelope by the definition above."""
    for K, n in ((5, 4096), (10, 4096)):
        res = _f32_bound_rollout(E, oracle, n, 1000, dict(sample_time=K * 0.01), 21)
        assert res["n_done"] == n * (1000 * K // 2000)
        _assert_bound(f"canonical K={K} {n}x1000", res, 1e-6, 2e-3, max_excused=0.01)
        assert np.quantile(res["obs"], 0.99) <= 3e-7


def test_f32_far_envelope_rare_paths(E, oracle):
    """Elevator commands held for 2..20 s put environments at high angles of attack, beyond +-90 deg of pitch
    (the DLL's asin fold) and above the tropopause: every fall-back of the f32 path (libm trigonometry outside the
    polynomial ranges, table interval re-searches, pitch fold) is exercised.  Inside the envelope the held-elevator
    trajectories keep a bound of 1e-4 / 5e-3 on every env (large, slowly varying elevator: the same force error acts in one
    direction for seconds); outside it outputs stay finite, done flags stay bit-exact, and even counting the tumbling
    phases the median env stays inside the canonical 1e-5 (measured round 1: median 1.5e-7, p99 2.9e-3, max 4.9e-3 with
    the elevator held for a whole episode)."""
    for K, n, hold in ((10, 512, 200), (5, 512, 40)):
        res = _f32_bound_rollout(E, oracle, n, 420, dict(sample_time=K * 0.01), 33, sticky=hold)
        _assert_bound(f"far-envelope K={K} hold={hold}", res, 1e-4, 5e-3, max_excused=0.9)
        q = np.quantile(res["obs_all"], [0.5, 0.9, 0.99])
        print(f"   incl. tumbling phases: per-env worst median {q[0]:.1e} p90 {q[1]:.1e} p99 {q[2]:.1e} max {res['obs_all'].max():.1e}")
        assert res["excused"] > 0          # the test really leaves the envelope
        assert q[0] <= 1e-5 and res["obs_all"].max() <= 0.2


# Per-family bounds of the f32 path: (|d obs| / (1 + |obs|), |d reward|, largest share of env-steps outside the envelope),
# every one asserted on ALL 512 envs at EVERY step inside the envelope.  Numbers = measured maxima (round 2,
# tools/family_probe.py / profiles/r2_family_bounds.md) with a margin of 3-4x.  Why the families differ:
#  * canonical dynamics (K10, K1, minimal, fixed aero error, TF reward): the float32 force error (~1e-6 relative per
#    evaluation) integrated over an episode -> 1e-6 on the normalised observation;
#  * action laws that feed U_com_PID back into the elevator (ADD_PROC, ADD_DIRECT) and the closed altitude loop
#    (SEMI_MANUAL / HYBRID): the PID's derivative path (Kd N ~ 390) turns a 1e-7 pitch error into ~2e-6 rad of elevator,
#    and a saturation / anti-windup event that falls on the other side of a model step shifts an integrator by Ki dv h
#    ~ 1e-3 rad for good -> 5e-4;
#  * PID_LIKE reward exp(-10 |U_com - U_com_PID| / 34 deg) reads that elevator difference directly -> 3e-2 on the reward.
FAMILY_BOUNDS = {
    "K10": (1e-6, 2e-3, 0.02),
    "K1_tk3": (1e-6, 2e-3, 0.02),
    "minimal": (1e-6, 2e-3, 0.02),
    "fixed_aero_err": (1e-6, 2e-3, 0.02),
    "tfref_unnormalised": (1e-5, 3e-3, 0.02),
    "pidaero_pidlike_limiter": (2e-6, 3e-2, 0.02),
    "speed_addproc": (3e-4, 5e-3, 0.02),
    "aero_adddirect_osc": (5e-4, 5e-3, 0.02),
    "quality_semimanual": (5e-4, 2e-3, 0.02),
    "state_angvel_hybrid_dist": (1e-4, 2e-3, 0.05),
}


@pytest.mark.parametrize("name", sorted(VARIANTS) + TUNED_F32)
def test_f32_variants_within_bound(E, oracle, name):
    fam, ekw = TUNED.get(name, (name, None))
    kw = VARIANTS.get(fam, {})
    steps = 320 if fam == "K1_tk3" else 420
    ob, rb, ex = FAMILY_BOUNDS["K10" if fam == "canonical" else fam]
    res = _f32_bound_rollout(E, oracle, 512, steps, kw, 9, ekw=ekw, params=tuned_params(oracle) if name in TUNED else None)
    assert res["n_done"] >= 512
    _assert_bound(name, res, ob, rb, max_excused=ex)


@pytest.mark.parametrize("dtype_name", ["F64", "F32"])
def test_config0_single_env_10k_steps(E, dtype_name):
    """BASELINE configs[0]: ONE environment, 10 000 env steps (50 000 model steps) of fixed-seed random elevator actions,
    against the digest of the trajectory the reference DLL produced (tests/golden/make_config0.py): episodic (25
    resets) and one 100 s flight (tk = 1e9; the f32 handle then runs with tick > 16383, the plain tick word)."""
    import sys
    sys.path.insert(0, HERE)
    from config0_check import check_config0
    g = json.load(open(os.path.join(HERE, "golden", "config0_golden.json")))
    dtype = getattr(E, dtype_name)
    a = np.random.default_rng(g["action_seed"]).uniform(-1.0, 1.0, g["n_steps"])
    for name, kw in (("episodic", {}), ("long_flight", dict(tk=1.0e9))):
        eng = E.BatchEngine(n_envs=1, dtype=dtype, seed=g["seed"], auto_reset=True, **kw)
        eng.reset()
        n = g["n_steps"]
        obs = np.zeros((n, 3)); rew = np.zeros(n); done = np.zeros(n, dtype=bool)
        term = np.zeros((1, 3), eng.np_dtype)
        for k in range(n):
            _, r, d, term = eng.step_host(a[k:k + 1], terminal_obs=term)
            obs[k], rew[k], done[k] = term[0], r[0], d[0]
        tol = (2e-9, 1e-9) if dtype == E.F64 else (1e-5, 2e-3)
        check_config0(g["cases"][name], obs, rew, done, *tol)
        eng.close()


def test_full_size_properties_config3(E, oracle):
    """BASELINE configs[2]: 1M envs, f32, K=10, in-kernel auto-reset -- size-independent properties."""
    import torch
    n, K = 1 << 20, 10
    kw = dict(sample_time=K * 0.01)
    eng = E.BatchEngine(n_envs=n, dtype=E.F32, seed=1, **kw)
    # both handles launch on torch's current stream, so the action generation / slicing below is ordered with the steps
    eng.use_stream(torch.cuda.current_stream().cuda_stream)
    act, obs, rew, done = eng.alloc_io()
    eng.reset(obs)
    eng.synchronize()
    assert float(obs.abs().max()) == 0.0
    gen = torch.Generator(device="cuda").manual_seed(0)
    # sharding invariance: a 4096-env handle holding the same GLOBAL env ids gives bit-identical results
    lo = 777 * 128
    sl = E.BatchEngine(n_envs=4096, dtype=E.F32, seed=1, env_id_offset=lo, **kw)
    sl.use_stream(torch.cuda.current_stream().cuda_stream)
    a2, o2, r2, d2 = sl.alloc_io()
    sl.reset(o2)
    # oracle on 512 of those envs
    ob = oracle.OracleBatch(oracle.make_cfg(seed=1, **kw), 512, env_id_offset=lo)
    ob.reset()
    total_done = 0
    ret_first_episode = 0.0
    for k in range(205):
        act.uniform_(-1, 1, generator=gen)
        eng.step(act, obs, rew, done)
        a2.copy_(act[lo:lo + 4096])
        sl.step(a2, o2, r2, d2)
        eng.synchronize(); sl.synchronize()
        assert torch.isfinite(obs).all() and torch.isfinite(rew).all()
        # CLASSIC reward range: r1..r4 in (0, 1]; rf >= -kf * (|dvartheta| / (2 |vf|)) with the folded pitch error
        # below 100 deg and |vf| >= 1 deg (env/ctrl_env.py:124-143)
        assert float(rew.min()) >= -5.0 and float(rew.max()) <= 1.0 + 1e-6
        assert torch.equal(obs[lo:lo + 4096], o2) and torch.equal(rew[lo:lo + 4096], r2)
        assert torch.equal(done[lo:lo + 4096], d2)
        nd = int(done.sum())
        # tk = 20 s at K = 10: every env finishes exactly at env step 200 (done <=> tick >= 2000), none before
        assert nd == (n if k == 199 else 0)
        total_done += nd
        if k < 200:
            ret_first_episode += float(rew.double().sum())
        o_o, r_o, d_o, _ = ob.step(act[lo:lo + 512].double().cpu().numpy())
        assert np.array_equal(d_o, done[lo:lo + 512].cpu().numpy().astype(bool))
        assert np.abs(obs[lo:lo + 512].double().cpu().numpy() - o_o).max() <= 1e-5
        assert np.abs(rew[lo:lo + 512].double().cpu().numpy() - r_o).max() <= 1e-3
        if k == 199:
            assert float(obs.abs().max()) == 0.0   # auto-reset returns the (all-zero) reset observation
    assert total_done == n
    # checksum of checksums: the in-kernel episode statistics equal the sums of the per-step outputs
    st = eng.episode_stats()
    assert st[0] == n and st[2] == 200.0 * n
    assert abs(st[1] - ret_first_episode) <= 1e-9 * abs(ret_first_episode)
    ret, ln = eng.last_episode()
    assert (ln == 200).all() and abs(ret.sum() - st[1]) <= 1e-9 * abs(st[1])
    # determinism: two fresh handles with the same seed replay the same step bit for bit
    outs = []
    for _ in range(2):
        e2 = E.BatchEngine(n_envs=n, dtype=E.F32, seed=1, **kw)
        e2.use_stream(torch.cuda.current_stream().cuda_stream)
        b_act, b_obs, b_rew, b_done = e2.alloc_io()
        e2.reset(b_obs)
        b_act.uniform_(-1, 1, generator=torch.Generator(device="cuda").manual_seed(0))
        e2.step(b_act, b_obs, b_rew, b_done)
        e2.synchronize()
        outs.append((b_obs.clone(), b_rew.clone()))
        e2.close()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
