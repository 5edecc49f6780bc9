"""GPU tests of the drop-in surfaces: the scalar model_simple.so boundary bound exactly as
core/model.py does, Model, Controller/ControllerEnv (gym API) and B747VecEnv (SB3 VecEnv contract)."""
import ctypes
import json
import math
import os
import sys
import random
import shutil
import tempfile

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)
DEG = math.pi / 180


def _kats():
    return json.load(open(os.path.join(HERE, "golden", "model_kats.json")))


def _tol(name):
    return {"dvartheta_dt_dt": (1e-6, 1e-9), "dvartheta_dt": (1e-8, 1e-11)}.get(name, (1e-9, 1e-12))


def test_scalar_boundary_bound_like_core_model_py():
    """core/model.py:99-164: copy the library, LoadLibrary, bind 3 functions + globals with in_dll."""
    from b747_rl_ctrl_b200 import _lib
    real_T = ctypes.c_double
    tmp = tempfile.mkdtemp()
    insts = []
    for k in range(2):  # two private copies == two independent Model instances
        path = os.path.join(tmp, f"copy{k}.so")
        shutil.copyfile(_lib.SCALAR_LIB_PATH, path)
        insts.append(ctypes.cdll.LoadLibrary(path))
    dll = insts[0]
    init, step = getattr(dll, "model_simple_initialize"), getattr(dll, "model_simple_step")
    state = (real_T * 6).in_dll(dll, "state")
    sim_time = real_T.in_dll(dll, "sim_time")
    use_ss = real_T.in_dll(dll, "use_PID_SS")
    dv = real_T.in_dll(dll, "dvartheta")
    use_ss.value = 1.0
    init()
    assert list(state) == [0.0] * 6 and sim_time.value == 0.0
    step()
    k1 = _kats()["K1"]["snaps"]
    assert sim_time.value == 0.01
    assert np.allclose(list(state), k1["1"]["state"], rtol=1e-12, atol=1e-13)
    assert dv.value == pytest.approx(k1["1"]["dvartheta"], rel=1e-12)
    for _ in range(4):
        step()
    assert np.allclose(list(state), k1["5"]["state"], rtol=1e-12, atol=1e-13)
    # the second copy is untouched (private globals, like one DLL copy per Model)
    assert real_T.in_dll(insts[1], "sim_time").value == 0.0
    shutil.rmtree(tmp, ignore_errors=True)


def test_scalar_boundary_tunables_match_oracle():
    """The scalar drop-in with every airframe parameter and gain away from its default, written into the exported
    globals the way core/model.py writes them (in_dll(...).value, array items), and both gain sets acting (use_PID_SS =
    use_PID_CS = 1): every exported signal against the oracle's model given the same values, 1e-9, over 300 steps."""
    from b747_rl_ctrl_b200 import _lib
    from oracle import oracle as O
    from test_gpu_parity import DDT2, SIG_FIELDS, tuned_params
    O.build()
    real_T = ctypes.c_double
    tmp = tempfile.mkdtemp()
    path = os.path.join(tmp, "tuned.so")
    shutil.copyfile(_lib.SCALAR_LIB_PATH, path)
    dll = ctypes.cdll.LoadLibrary(path)
    m = O.CModel()

    def glob(name, n=1):
        return (real_T * n).in_dll(dll, name) if n > 1 else real_T.in_dll(dll, name)

    def put(name, v):
        v = np.atleast_1d(np.asarray(v, np.float64))
        if len(v) > 1:
            arr = glob(name, len(v))
            for k, x in enumerate(v):
                arr[k] = float(x)
        else:
            glob(name).value = float(v[0])
        m.set(name, v if len(v) > 1 else v[0])

    for nm, v in tuned_params(O).items():
        put(nm, v)
    put("state0", [0.0, 8000.0, 230.0, 2.0, 0.02, 0.0])
    dll.model_simple_initialize()
    m.initialize()
    for nm, v in (("use_PID_SS", 1.0), ("use_PID_CS", 1.0), ("h_zh", 8200.0), ("vartheta", 0.0), ("deltaz", 0.0)):
        put(nm, v)
    state = glob("state", 6)
    worst = {}
    for k in range(300):
        dll.model_simple_step()
        m.step()
        for name, (oname, idx, floor) in SIG_FIELDS.items():
            ref = np.atleast_1d(m.get(oname))[idx]
            got = state[idx] if oname == "state" else glob(oname).value
            q = abs(got - ref) / max(1e-9 * (abs(ref) + floor), 1e-300)
            worst[oname + str(idx)] = max(worst.get(oname + str(idx), 0.0), q)
        _, oname, a, r = DDT2
        ref = m.get(oname)
        worst[oname] = max(worst.get(oname, 0.0), abs(glob(oname).value - ref) / (a + r * abs(ref)))
    print("scalar drop-in, worst signals (deviation / bar):", sorted(worst.items(), key=lambda kv: -kv[1])[:4])
    assert all(v <= 1.0 for v in worst.values()), {k: v for k, v in worst.items() if not v <= 1.0}
    assert glob("sim_time").value == pytest.approx(3.0) and abs(glob("U_com_PID").value) > 0
    shutil.rmtree(tmp, ignore_errors=True)


@pytest.mark.parametrize("name", ["K1", "K3", "K4", "K5"])
def test_model_dropin_matches_dll_kats(name):
    """Model attribute surface (core/model.py) stepping on the GPU vs signals recorded from the DLL."""
    from b747_rl_ctrl_b200.core.model import Model
    case = _kats()[name]
    p = case["params"]
    m = Model(use_PID_SS=bool(p.get("use_PID_SS", 0)), use_PID_CS=bool(p.get("use_PID_CS", 0)),
              initial_state=np.array(p["state0"]) if "state0" in p else None)
    assert (m.state == 0).all() and m.time == 0.0 and m.step_num == -1
    if "h_zh" in p:
        m.hzh = p["h_zh"]
    if "aero_err" in p:
        m.aero_err = np.array(p["aero_err"])
    m.vartheta_zh = p.get("vartheta", 5 * DEG if name == "K1" else 0.0)
    if name == "K1":
        m.vartheta_zh = 0.08726646259971647  # DLL default of `vartheta` (Model.initialize zeroes it)
    rng = random.Random(0)
    steps = min(case["steps"], 1300)
    py2sig = {"time": "sim_time", "vartheta_ref": "vartheta_zh", "deltaz_ref": "U_com_PID", "deltaz_com": "U_com",
              "deltaz_real": "deltaz_RP", "Kalpha": "K_alpha"}
    for k in range(steps):
        if case["elevator"] and k % 5 == 0:
            m.deltaz = rng.uniform(-0.2967, 0.2967)
        m.step()
        snap = case["snaps"].get(str(k + 1))
        if snap is None:
            continue
        assert np.allclose(m.state, snap["state"], rtol=1e-9, atol=1e-12), (name, k + 1)
        for attr in ["time", "vartheta_ref", "deltaz_ref", "deltaz_com", "deltaz_real", "CXa", "CYa", "mz", "Kalpha",
                     "dCm_ddeltaz", "dvartheta", "dvartheta_int", "dvartheta_dt", "dvartheta_dt_dt", "TAE", "ITAE",
                     "TSE", "ITSE", "AE", "IAE", "SE", "ISE"]:
            sig = py2sig.get(attr, attr)
            rel, ab = _tol(sig)
            assert np.allclose(getattr(m, attr), snap[sig], rtol=rel, atol=ab), (name, k + 1, attr)
    assert m.step_num == steps - 1
    assert set(m.state_dict) == {"x", "y", "Vx", "Vy", "vartheta", "wz"}


def test_controller_env_k7():
    """SURVEY.md 8c K7 through the ControllerEnv drop-in (gym API), float64."""
    from b747_rl_ctrl_b200.core.controller import CtrlMode, CtrlType
    from b747_rl_ctrl_b200.env.ctrl_env import ControllerEnv, ObservationType, RewardType
    g = np.load(os.path.join(HERE, "golden", "env_golden.npz"))
    env = ControllerEnv(ObservationType.PID_LIKE, RewardType.CLASSIC, True, True, CtrlType.MANUAL, CtrlMode.DIRECT_CONTROL,
                        tk=20, reset_ref_mode=None, sample_time=0.05, use_limiter=False, action_max=17 * DEG)
    assert env.observation_space.shape == (3,) and env.action_space.shape == (1,)
    env.ctrl.vartheta_func = lambda _: 5 * DEG
    obs = env.reset(np.array([0, 11000, 250, 0, 0, 0]))
    assert list(obs) == [0.0, 0.0, 0.0]
    rng = random.Random(0)
    ret = 0.0
    for k in range(400):
        a = np.array([rng.uniform(-1, 1)])
        a0 = a[0]
        obs, r, done, info = env.step(a)
        assert a[0] == a0 * (17 * DEG)          # the reference scales the caller's array in place
        assert np.allclose(obs, g["k7/obs"][k], rtol=1e-9, atol=2e-12), k
        assert abs(r - g["k7/rew"][k]) <= 1e-9
        assert done == (k == 399) and info == {}
        ret += r
    assert ret == pytest.approx(218.4897443782656, abs=1e-8)
    assert env.ctrl.is_done and env.is_done()
    assert env.ctrl.model.time == 20.0
    assert env.ctrl.vartheta_ref == 5 * DEG
    q = env.ctrl.quality()
    assert 0 < q < 1
    # ADD_PROC with a = 0 is the pure PID loop; its return is the published-curve anchor of SURVEY.md 6
    env = ControllerEnv(ObservationType.PID_LIKE, RewardType.CLASSIC, True, True, CtrlType.MANUAL, CtrlMode.ADD_PROC_CONTROL,
                        tk=20, reset_ref_mode=None, sample_time=0.05, action_max=1.0)
    env.ctrl.vartheta_func = lambda _: 5 * DEG
    env.reset(np.array([0, 11000, 250, 0, 0, 0]))
    ret = sum(env.step(np.array([0.0]))[1] for _ in range(400))
    assert ret == pytest.approx(365.092282070656, abs=1e-8)


def test_vec_env_contract(oracle):
    """SB3 VecEnv duck type: shapes, auto-reset observation, terminal_observation, episode info."""
    from b747_rl_ctrl_b200.vec_env import B747VecEnv
    from b747_rl_ctrl_b200 import engine as E
    n = 64
    venv = B747VecEnv(n, tk=0.5, sample_time=0.05, seed=4, dtype=E.F64)  # 10-step episodes
    assert venv.num_envs == n and venv.observation_space.shape == (3,) and venv.action_space.shape == (1,)
    obs = venv.reset()
    assert obs.shape == (n, 3) and (obs == 0).all()
    ob = oracle.OracleBatch(oracle.make_cfg(tk=0.5, seed=4), n)
    ob.reset()
    rng = np.random.default_rng(1)
    for k in range(25):
        a = rng.uniform(-1, 1, (n, 1))
        venv.step_async(a)
        obs, rew, dones, infos = venv.step_wait()
        o_o, r_o, d_o, t_o = ob.step(a[:, 0])
        assert obs.shape == (n, 3) and rew.shape == (n,) and dones.dtype == bool and len(infos) == n
        assert np.array_equal(dones, d_o) and np.allclose(obs, o_o, rtol=1e-9, atol=2e-9) and np.allclose(rew, r_o, atol=1e-9)
        if (k + 1) % 10 == 0:
            assert dones.all() and (obs == 0).all()
            for i in range(n):
                assert np.allclose(infos[i]["terminal_observation"], t_o[i], rtol=1e-9, atol=2e-9)
                assert infos[i]["episode"]["l"] == 10 and infos[i]["episode"]["r"] > 0
        else:
            assert not dones.any() and infos[0] == {}
    assert venv.env_is_wrapped(None) == [False] * n and venv.seed(1) == [1 + i for i in range(n)]
    st = venv.episode_stats()
    assert st[0] == 2 * n and st[2] == 20 * n
    venv.close()


@pytest.mark.parametrize("n,mode", [(1000, -1), (1000, 0), (1000, 1), (200000, -1), (200000, 0), (777, "pageable"),
                                    (5000, "chunked")])
def test_packed_host_step_equals_plain_step(n, mode):
    """b747_step_host_packed (one float4 record per env + done bits; zero-copy on pinned buffers, staged copies
    otherwise) returns exactly what b747_step_host returns: record = (terminal observation, reward), bit = done.
    "chunked": staged copies (mode 0) pipelined over set_host_chunks(7) chunks, below the automatic chunking's size."""
    import torch
    from b747_rl_ctrl_b200 import engine as E
    kw = dict(dtype=E.F32, seed=6, sample_time=0.05, tk=0.35)  # 7-step episodes: auto-resets inside the run
    ref, pk = E.BatchEngine(n_envs=n, **kw), E.BatchEngine(n_envs=n, **kw)
    ref.reset(); pk.reset()
    nw = (n + 31) // 32
    if mode == "pageable":
        act, out4, bits = np.zeros(n, np.float32), np.zeros((n, 4), np.float32), np.zeros(nw, np.uint32)
    else:
        if mode == "chunked":
            pk.set_host_chunks(7)
        pk.set_host_mode(0 if mode == "chunked" else mode)
        keep = [torch.zeros(n).pin_memory(), torch.zeros(n, 4).pin_memory(), torch.zeros(nw, dtype=torch.int32).pin_memory()]
        act, out4, bits = keep[0].numpy(), keep[1].numpy(), keep[2].numpy().view(np.uint32)
    rng = np.random.default_rng(2)
    term = np.zeros((n, 3), np.float32)
    n_done = 0
    for k in range(16):
        a = rng.uniform(-1, 1, n).astype(np.float32)
        _, rew, done, term = ref.step_host(a, terminal_obs=term)
        act[:] = a
        out4[:] = -7.0
        bits[:] = 0xdeadbeef
        pk.step_host_packed(act, out4, bits)
        d = np.unpackbits(bits.view(np.uint8), bitorder="little")[:n]
        assert np.array_equal(d, done), k
        assert np.array_equal(out4[:, :3], term) and np.array_equal(out4[:, 3], rew), k
        n_done += int(done.sum())
    assert n_done == 2 * n
    if mode == "chunked":
        per = -(-(-(-n // 7)) // 128) * 128  # whole thread blocks per chunk
        assert pk.launch_count - ref.launch_count == 16 * (-(-n // per) - 1)
    s0, s1 = ref.episode_stats(), pk.episode_stats()
    assert s0[0] == s1[0] == 2 * n and np.allclose(s0, s1, rtol=1e-12)
    for name in ("h", "th", "tick", "ep_idx", "ep_return"):
        assert np.array_equal(ref.get(name), pk.get(name)), name
    # device-buffer form
    act_d, out_d = torch.zeros(n, device="cuda"), torch.zeros(n, 4, device="cuda")
    bits_d = torch.zeros(nw, dtype=torch.int32, device="cuda")
    a = rng.uniform(-1, 1, n).astype(np.float32)
    _, rew, done, term = ref.step_host(a, terminal_obs=term)
    act_d.copy_(torch.from_numpy(a))
    pk.step_packed(act_d, out_d, bits_d)
    pk.synchronize()
    assert np.array_equal(out_d.cpu().numpy()[:, 3], rew) and np.array_equal(out_d.cpu().numpy()[:, :3], term)
    ref.close(); pk.close()


@pytest.mark.parametrize("obs_type,od,R", [(1, 5, 8), (4, 7, 8), (2, 8, 12), (3, 10, 12)])
def test_packed_records_of_wider_observation_layouts(obs_type, od, R):
    """Records are 4 * ceil((obs_dim + 1) / 4) floats: observation, reward, zero padding -- for every layout."""
    import torch
    from b747_rl_ctrl_b200 import engine as E
    n = 1500
    kw = dict(dtype=E.F32, seed=6, sample_time=0.05, tk=0.35, obs_type=obs_type)
    ref, pk = E.BatchEngine(n_envs=n, **kw), E.BatchEngine(n_envs=n, **kw)
    assert pk.record_floats == R and pk.obs_dim == od
    ref.reset(); pk.reset()
    keep = [torch.zeros(n).pin_memory(), torch.zeros(n, R).pin_memory(), torch.zeros((n + 31) // 32, dtype=torch.int32).pin_memory()]
    act, out, bits = keep[0].numpy(), keep[1].numpy(), keep[2].numpy().view(np.uint32)
    rng = np.random.default_rng(2)
    term = np.zeros((n, od), np.float32)
    for k in range(9):
        a = rng.uniform(-1, 1, n).astype(np.float32)
        _, rew, done, term = ref.step_host(a, terminal_obs=term)
        act[:] = a
        out[:] = -7.0
        pk.step_host_packed(act, out, bits)
        assert np.array_equal(np.unpackbits(bits.view(np.uint8), bitorder="little")[:n], done), k
        assert np.array_equal(out[:, :od], term) and np.array_equal(out[:, od], rew) and (out[:, od + 1:] == 0).all(), k
    assert done.sum() == 0 and ref.episode_stats()[0] == n
    ref.close(); pk.close()


def test_packed_step_rejected_where_it_does_not_apply():
    from b747_rl_ctrl_b200 import engine as E
    e = E.BatchEngine(n_envs=64, dtype=E.F64)
    with pytest.raises(E.B747Error):
        e.step_host_packed(np.zeros(64, np.float32), np.zeros((64, 4), np.float32), np.zeros(2, np.uint32))
    e.close()


@pytest.mark.parametrize("copy_outputs", [True, False])
def test_vec_env_under_sb3_standin(oracle, copy_outputs):
    """The numpy-mode VecEnv (packed zero-copy path) driven the way stable-baselines3 drives it: float32 [N, 1] actions
    through step_async / step_wait inside a VecMonitor, in collect_rollouts' call order (an observation is read once
    more after the NEXT step returned).  Checked against the oracle: observations (zero where an env finished),
    rewards, dones, terminal observations, and the episode records of both the env's own monitor and VecMonitor."""
    import sb3_standin as sb3
    from b747_rl_ctrl_b200.vec_env import B747VecEnv
    n = 300
    venv = B747VecEnv(n, tk=0.5, sample_time=0.05, seed=4, copy_outputs=copy_outputs)  # f32, 10-step episodes
    assert sb3.conforms(venv) == []
    env = sb3.VecMonitor(venv)
    assert env.seed(4) == [4 + i for i in range(n)]
    obs = env.reset()
    assert obs.shape == (n, 3) and obs.dtype == np.float32 and (obs == 0).all()
    ob = oracle.OracleBatch(oracle.make_cfg(tk=0.5, seed=4), n)
    ob.reset()
    rng = np.random.default_rng(1)
    roll = sb3.collect_rollouts(env, lambda o: rng.uniform(-1.2, 1.2, (n, 1)), 25, obs)   # some actions get clipped
    assert roll["obs"].shape == (25, n, 3) and roll["done"].dtype == bool
    rets = np.zeros(n)
    k_term = 0
    for k in range(25):
        a = np.clip(roll["act"][k][:, 0], -1, 1).astype(np.float64)
        o_o, r_o, d_o, t_o = ob.step(a)
        rets += r_o
        assert np.array_equal(roll["done"][k], d_o)
        assert np.abs(roll["rew"][k] - r_o).max() <= 1e-3
        nxt = roll["obs"][k + 1] if k + 1 < 25 else roll["last_obs"]
        assert np.abs(nxt - o_o).max() <= 1e-5, k              # what collect_rollouts stored one step later
        if d_o.any():
            assert d_o.all() and (nxt == 0).all()
            for i in range(n):
                j, tobs, epi = roll["terminal"][k_term]
                k_term += 1
                assert j == i and np.abs(tobs - t_o[i]).max() <= 1e-5
                assert epi["l"] == 10 and abs(epi["r"] - rets[i]) <= 1e-2
            rets[:] = 0
    assert k_term == 2 * n
    venv.close()


def test_vec_env_per_env_views(oracle):
    """get_attr / set_attr / env_method address single environments (what SubprocVecEnv forwards to its workers):
    `env.get_attr('ctrl')[0].storage.storage` (neural/setups.py:216), `env.ctrl.vartheta_func = lambda _: ref`,
    `ctrl.quality()`, `envs[i].reset(state0)`; seed(s) re-keys the Philox stream of later resets."""
    from b747_rl_ctrl_b200.vec_env import B747VecEnv
    from b747_rl_ctrl_b200 import engine as E
    n = 8
    venv = B747VecEnv(n, tk=2.0, sample_time=0.05, seed=3, dtype=E.F64, record_capacity=260, export_signals=True)
    venv.reset()
    ctrls = venv.get_attr("ctrl")
    assert len(ctrls) == n and ctrls[0] is venv.ctrl and ctrls[3] is venv.envs[3].ctrl
    assert venv.get_attr("ctrl", indices=[2, 5])[1] is ctrls[5]
    assert venv.get_attr("norm_obs") == [True] * n and venv.get_attr("tk", indices=1) == [2.0]
    # re-target env 2 and restart env 5 from an explicit state, leave the others alone
    ctrls[2].vartheta_func = lambda _: 4 * DEG
    h_before = venv.engine.get("h")
    ctrls[5].vartheta_func = lambda _: -3 * DEG
    venv.env_method("reset", np.array([0, 9000, 240, 0, 0, 0]), indices=[5])
    h_after = venv.engine.get("h")
    assert h_after[5] == 9000.0 and np.array_equal(np.delete(h_after, 5), np.delete(h_before, 5))
    assert ctrls[2].vartheta_ref == 4 * DEG and ctrls[5].vartheta_ref == -3 * DEG
    rng = np.random.default_rng(0)
    for k in range(7):
        obs, rew, dones, infos = venv.step(rng.uniform(-1, 1, (n, 1)))
    st = ctrls[5].storage.storage                       # Controller.storage: one record per MODEL step
    assert len(st["t"]) == 35 and st["t"][-1] == pytest.approx(0.35) and st["y"][0] == pytest.approx(9000.0, abs=5)
    assert set(st) >= {"t", "U_com", "U_PID", "deltaz", "hzh", "vartheta_ref", "U_RL", "x", "y", "Vx", "Vy", "vartheta", "wz"}
    assert st["vartheta_ref"][-1] == pytest.approx(-3.0)
    q = ctrls[2].quality()
    assert 0 < q <= 1 and q == pytest.approx(math.exp(-6 * ctrls[2].model.ITSE / (2.0 * (4 * DEG) ** 2)))
    assert venv.env_method("get_reward", indices=[1]) == [pytest.approx(float(rew[1]))]
    assert np.allclose(venv.get_attr("state_box", indices=[4])[0], obs[4])
    assert ctrls[0].model.time == pytest.approx(0.35) and not ctrls[0].is_done
    with pytest.raises(NotImplementedError):
        ctrls[1].vartheta_func = lambda t: 0.01 * t   # the batched kernels hold a reference constant over an episode
    # seed(s): later random resets draw from the re-keyed stream, identically to a handle built with that seed
    venv.seed(11)
    venv.env_method("reset", indices=[0, 1])
    other = E.BatchEngine(n_envs=n, dtype=E.F64, seed=11, tk=2.0)
    other.set("ep_idx", venv.engine.get("ep_idx") - np.array([1, 1] + [0] * (n - 2)))
    other.reset()
    assert np.array_equal(other.get("h")[:2], venv.engine.get("h")[:2])
    assert not np.array_equal(venv.engine.get("h")[:2], h_before[:2])
    other.close()
    venv.close()


def test_controller_time_varying_reference_function():
    """Controller(vartheta_func=<any callable>): the reference is func(model.time) written before every env step
    (core/controller.py:233-236).  A 3-sine Python function must reproduce the in-kernel oscillating reference."""
    from b747_rl_ctrl_b200.core.controller import Controller, CtrlMode, CtrlType
    from b747_rl_ctrl_b200 import engine as E
    A, f = [3 * DEG, 2 * DEG, 1 * DEG], [0.05, 0.2, 0.4]
    func = lambda t: sum(a * math.sin(2 * math.pi * w * t) for a, w in zip(A, f))
    c = Controller(CtrlType.MANUAL, CtrlMode.DIRECT_CONTROL, tk=3.0, sample_time=0.05, vartheta_func=func)
    c.reset(np.array([0, 9000, 230, 2, 0, 0]))
    ref = E.BatchEngine(n_envs=1, dtype=E.F64, reset_ref_mode=E.RESET_NONE, tk=3.0, sample_time=0.05, norm_act=False,
                        auto_reset=False)
    ref.reset_to([E.episode([0, 9000, 230, 2, 0, 0], osc=(A, f))])
    rng = np.random.default_rng(5)
    for k in range(60):
        a = rng.uniform(-0.2, 0.2, 1)
        c.step(a)
        o_r, r_r, d_r = ref.step_host(a)
        obs, rew, done = c._last
        assert np.abs(obs - o_r[0]).max() <= 1e-11 and abs(rew - r_r[0]) <= 1e-10 and done == bool(d_r[0]), k
        assert c.vartheta_ref == pytest.approx(func(k * 0.05), abs=1e-15)
    assert done and abs(obs[1]) > 1e-4
    # altitude reference through the СУ PID: h_func(t) is written to h_zh when the altitude loop is closed
    c2 = Controller(CtrlType.SEMI_MANUAL, CtrlMode.ADD_PROC_CONTROL, tk=2.0, sample_time=0.05, action_max=1.0,
                    h_func=lambda t: 11000.0 + 20.0 * t)
    c2.reset(np.array([0, 11000, 250, 0, 0, 0]))
    for k in range(10):
        c2.step(np.array([0.0]))
    assert c2.model.hzh == pytest.approx(11000.0 + 20.0 * 0.45)
    ref.close()


def test_controller_draws_aero_disturbance_on_every_reset():
    """core/controller.py:181-191: DisturbanceMode.AERO_DISTURBANCE without a fixed aero_err draws a fresh Gaussian error
    from numpy's global stream on every reset, also when the reset itself is deterministic (reset_ref_mode None)."""
    from b747_rl_ctrl_b200.core.controller import Controller, CtrlMode, CtrlType, DisturbanceMode
    c = Controller(CtrlType.MANUAL, CtrlMode.DIRECT_CONTROL, disturbance_mode=DisturbanceMode.AERO_DISTURBANCE, tk=1.0,
                   vartheta_func=lambda _: 0.05)
    np.random.seed(0)
    want = [np.array([np.random.normal(m, 0.5) for m in (-0.1, 0.1, -0.1, -0.1, 0.1)]) for _ in range(2)]
    np.random.seed(0)
    for k in range(2):
        c.reset(np.array([0, 11000, 250, 0, 0, 0]))
        assert np.allclose(c.model.aero_err, want[k], rtol=0, atol=0)
    c.step(np.array([0.01]))
    assert c.model.CYa != 0.0


def test_vec_env_device_tensors():
    import torch
    from b747_rl_ctrl_b200.vec_env import B747VecEnv
    venv = B747VecEnv(4096, device_tensors=True)
    obs = venv.reset()
    assert obs.is_cuda and obs.shape == (4096, 3)
    a = torch.zeros(4096, 1, device="cuda")
    for _ in range(3):
        obs, rew, dones, infos = venv.step(a)
    assert obs.is_cuda and rew.is_cuda and dones.dtype == torch.bool and float(rew.min()) > 0
    venv.close()
    # episodes finishing on the device path: terminal observations are device tensors, monitor records host floats
    venv = B747VecEnv(256, device_tensors=True, tk=0.5, sample_time=0.05, seed=2)
    venv.reset()
    a = torch.zeros(256, 1, device="cuda")
    for k in range(12):
        last = venv._obs_d.clone()
        obs, rew, dones, infos = venv.step(a)
        if k == 9:
            assert bool(dones.all()) and float(obs.abs().max()) == 0.0
            assert all(i["terminal_observation"].is_cuda and i["episode"]["l"] == 10 and i["episode"]["r"] > 0 for i in infos)
            assert float(infos[7]["terminal_observation"].abs().max()) > 0
        else:
            assert not bool(dones.any()) and infos[7] == {}
    venv.close()


def test_reset_mask_and_reset_to():
    from b747_rl_ctrl_b200 import engine as E
    import torch
    n = 256
    eng = E.BatchEngine(n_envs=n, dtype=E.F64, seed=2)
    act, obs, rew, done = eng.alloc_io()
    eng.reset(obs)
    for _ in range(7):
        eng.step(act, obs, rew, done)
    eng.synchronize()
    assert (eng.get("tick") == 35).all()
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mask[::2] = 1
    h_before = eng.get("h")
    eng.reset(obs, mask=mask)
    eng.synchronize()
    t = eng.get("tick")
    assert (t[::2] == 0).all() and (t[1::2] == 35).all()
    assert (eng.get("ep_idx")[::2] == 2).all() and (eng.get("ep_idx")[1::2] == 1).all()
    assert np.array_equal(eng.get("h")[1::2], h_before[1::2])
    # explicit episodes (Controller.reset(state0) with a reference)
    e2 = E.BatchEngine(n_envs=2, dtype=E.F64, reset_ref_mode=E.RESET_NONE)
    e2.reset_to([E.episode([0, 11000, 250, 0, 0, 0], vref=5 * DEG), E.episode([10, 3000, 150, 5, 0.02, 0.001], vref=-3 * DEG)])
    assert list(e2.get("h")) == [11000.0, 3000.0] and list(e2.get("vref")) == [5 * DEG, -3 * DEG]
    assert np.allclose(e2.get("q3"), [0.0, math.sin(0.01)]) and list(e2.get("tick")) == [0, 0]


@pytest.mark.parametrize("dtype_name,n", [("F32", 5000), ("F64", 1300)])
def test_step_host_pipeline_equals_one_launch(dtype_name, n):
    """b747_step_host's chunked copy/compute pipeline returns bit-identical results to the one-launch form
    (ragged last chunk, auto-reset inside the run, terminal observations)."""
    from b747_rl_ctrl_b200 import engine as E
    dtype = getattr(E, dtype_name)
    engs = [E.BatchEngine(n_envs=n, dtype=dtype, seed=5, sample_time=0.05, tk=0.4) for _ in range(2)]
    engs[0].set_host_chunks(1)
    engs[1].set_host_chunks(7)
    for e in engs:
        e.reset()
    rng = np.random.default_rng(1)
    for k in range(20):
        a = rng.uniform(-1, 1, n)
        res = []
        for e in engs:
            term = np.zeros((n, e.obs_dim), e.np_dtype)
            res.append(e.step_host(a, terminal_obs=term))
        for x, y in zip(res[0], res[1]):
            assert np.array_equal(x, y), k
    assert res[0][2].any() or k > 8
    s0, s1 = engs[0].episode_stats(), engs[1].episode_stats()  # float64 atomics: summation order differs
    assert s0[0] == s1[0] and s0[2] == s1[2] and np.allclose(s0, s1, rtol=1e-12)
    per = -(-(-(-n // 7)) // 128) * 128  # whole thread blocks per chunk
    assert engs[1].launch_count - engs[0].launch_count == 20 * (-(-n // per) - 1)
    for e in engs:
        e.close()


def test_explicit_oscillating_episode_on_canonical_f32_handle(oracle):
    """b747_reset_to with an oscillating reference on a handle whose configuration family never draws one: the f32
    launch must leave the canonical (LEAN) kernel tier -- which has no reference generator -- for the full one."""
    from b747_rl_ctrl_b200 import engine as E
    n = 64
    kw = dict(sample_time=0.05, tk=3.0)
    eng = E.BatchEngine(n_envs=n, dtype=E.F32, seed=4, auto_reset=False, **kw)
    ob = oracle.OracleBatch(oracle.make_cfg(seed=4, **kw), n)
    osc = ([3 * DEG, 2 * DEG, 1 * DEG], [0.05, 0.2, 0.4])
    eps_g = [E.episode([0, 9000 + 10 * i, 230, 2, 0, 0], osc=osc) for i in range(n)]
    eps_o = [oracle.episode([0, 9000 + 10 * i, 230, 2, 0, 0], osc=osc) for i in range(n)]
    eng.reset_to(eps_g)
    ob.reset_to(eps_o)
    rng = np.random.default_rng(3)
    for k in range(60):
        a = rng.uniform(-1, 1, n).astype(np.float32)
        obs, rew, done = eng.step_host(a)
        o_o, r_o, d_o, _ = ob.step(a.astype(np.float64), auto_reset=False)
        assert np.array_equal(done.astype(bool), d_o)
        assert np.abs(obs - o_o).max() <= 1e-5 and np.abs(rew - r_o).max() <= 2e-3, k
    assert np.abs(o_o[:, 1]).max() > 1e-3  # the reference really moved
    eng.close()


def test_step_host_graph_replay_with_pinned_buffers():
    """With pinned host buffers b747_step_host replays its pipeline as a CUDA graph (one launch call per step); results
    equal the eager pipeline's on pageable buffers, across buffer sets and across parameter changes: set_param, entering
    per-env mode with a range, per-env values (device rows only) and another range, each redrawn at the 10-step
    episodes' auto-resets."""
    import torch
    from b747_rl_ctrl_b200 import engine as E
    n = 3000
    engs = [E.BatchEngine(n_envs=n, dtype=E.F32, seed=8, sample_time=0.05, tk=0.5) for _ in range(2)]
    for e in engs:
        e.set_host_chunks(4)
        e.reset()
    pin = lambda *shape, dt=torch.float32: torch.empty(*shape, dtype=dt).pin_memory()
    acts = [pin(n) for _ in range(3)]
    obs_p, rew_p, done_p = pin(n, 3), pin(n), pin(n, dt=torch.uint8)
    rng = np.random.default_rng(2)
    for k in range(40):
        for e in engs:
            if k == 12:  # launch arguments change: the captured graphs must not be replayed
                e.set_param("P", [2.0e5])
            elif k == 16:  # per-env mode: the twin kernel and its by-value EnvParams
                e.set_env_param_range("m0", [2.4e5], [3.4e5])
            elif k == 23:  # device rows only
                e.set_env_param("Iz", np.linspace(5.5e7, 7.5e7, n))
            elif k == 27:  # another by-value EnvParams
                e.set_env_param_range("PID_SS", [-6.5, -1.4, -7.0, 50.0], [-5.5, -1.1, -6.0, 65.0])
        a = rng.uniform(-1, 1, n).astype(np.float32)
        o0, r0, d0 = engs[0].step_host(a)
        buf = acts[k % 3]
        buf.copy_(torch.from_numpy(a))
        engs[1].step_host(buf.numpy(), obs_p.numpy(), rew_p.numpy(), done_p.numpy())
        assert np.array_equal(o0, obs_p.numpy()) and np.array_equal(r0, rew_p.numpy()) and np.array_equal(d0, done_p.numpy()), k
    assert engs[0].launch_count == engs[1].launch_count
    for e in engs:
        e.close()


def test_ppo_learns_on_gpu_vecenv():
    """BASELINE configs[4] in miniature: PPO (SB3-default hyper-parameters restated in torch) on 8192 GPU environments
    improves the episode return well beyond the untrained policy within a few seconds."""
    from b747_rl_ctrl_b200 import ppo
    r = ppo.train(n_envs=8192, threshold=None, total_steps=8192 * 32 * 40, max_seconds=120, seed=3)
    first, last = r["history"][0][2], r["history"][-1][2]
    print(f"PPO 8192 envs: ep_rew_mean {first:.1f} -> {last:.1f} in {r['seconds']:.1f} s ({r['steps_per_s']:.3e} steps/s)")
    assert last > first + 40 and last > 170
