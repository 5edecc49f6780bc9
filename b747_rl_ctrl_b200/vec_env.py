"""B747VecEnv -- the batched GPU environment with the stable-baselines3 VecEnv contract that
neural/agent.py:63-81 consumes (num_envs, observation_space, action_space, reset, step_async /
step_wait, close, seed, get_attr / set_attr / env_method / env_is_wrapped), replacing
SubprocVecEnv([ControllerEnv]*4) + VecMonitor: on done the returned observation is the reset
observation, infos[i]["terminal_observation"] holds the last one and infos[i]["episode"] the
{"r", "l", "t"} record VecMonitor would add.

Per-environment views: `env.envs[i]` is a ControllerEnv-shaped view of environment i and `env.envs[i].ctrl` a
Controller-shaped one (`model`, `storage`, `quality()`, `vartheta_ref`, `vartheta_func = lambda _: c`, ...), so the
calls the reference makes on its vectorised env -- `env.get_attr('ctrl')[0].storage.storage` (neural/setups.py:216),
`env.env_method(...)`, `env.set_attr(...)` -- address single environments like SubprocVecEnv's do.  `env.ctrl` is
environment 0's (the reference's callbacks hold a single env and read `env.ctrl`, neural/callbacks.py:61-64).

Two I/O modes:
  * numpy (default; what SB3 passes): pinned host buffers.  f32 handles take the packed zero-copy path
    (b747_step_host_packed: the kernel reads the actions from and stores one (obs, reward) record per env into the pinned
    buffers, done flags come back as one bit per env); float64 handles go through b747_step_host;
  * torch device tensors (`device_tensors=True`): obs/rew/done stay in HBM, for GPU-resident policies.

When stable-baselines3 is importable the class derives from its `VecEnv`, so `PPO('MlpPolicy', env)` takes it as is
(`BaseAlgorithm._wrap_env` wraps anything that is not a `VecEnv` instance into a DummyVecEnv).
"""
import math
import time

import numpy as np

from . import engine as E
from .env.ctrl_env import ObservationType, RewardType, make_spaces
from .core.controller import CtrlMode, CtrlType
from .tools.general import Storage, calc_stepinfo


try:  # a real SB3 VecEnv where SB3 exists (not in this image: no network), a duck type otherwise
    from stable_baselines3.common.vec_env import VecEnv as _VecEnvBase
except Exception:
    _VecEnvBase = object


def _pinned(shape, dtype):
    """Page-locked numpy array (a view of a pinned torch tensor, kept alive by the returned pair); pageable if torch
    cannot pin here."""
    try:
        import torch
        t = torch.zeros(shape, dtype=getattr(torch, np.dtype(dtype).name)).pin_memory()
        return t.numpy(), t
    except Exception:
        return np.zeros(shape, dtype), None


def th_index(t, idx):
    import torch
    return torch.as_tensor(idx, device=t.device, dtype=torch.long)


def _val(x, default=None):
    if x is None:
        return default
    return x.value if hasattr(x, "value") else int(x)


class _FieldModel:
    """Model-shaped view of env `i` of a throughput (f32) handle: the state fields the handle keeps (core/model.py:226
    labels).  Evaluation handles (export_signals=True) get the full ModelView instead."""
    labels = ['x', 'y', 'Vx', 'Vy', 'vartheta', 'wz']
    dt = 0.01

    def __init__(self, engine, i):
        self._e, self._i = engine, i

    def _g(self, name):
        return float(self._e.get(name)[self._i])

    @property
    def time(self):
        return self._g("tick") * self.dt

    @property
    def state(self):
        f32 = self._e.dtype == E.F32
        th = self._g("th") if f32 else 2.0 * math.atan2(self._g("q3"), self._g("q0"))
        return np.nan_to_num(np.array([self._g("x"), self._g("h"), self._g("Vx"), self._g("Vy"), th, self._g("wz")]))

    @property
    def state_dict(self):
        st = self.state
        return dict(zip(self.labels, st))

    @property
    def ITSE(self):
        return self._g("itse")

    @property
    def deltaz(self):
        return self._g("deltaz")

    @property
    def deltaz_ref(self):
        return self._g("sig_upid")

    @property
    def vartheta_zh(self):
        return self._g("vref")

    @property
    def hzh(self):
        return self._g("href") if self._e.dtype == E.F32 else self._g("h_zh")


class VecCtrlView:
    """Controller-shaped view of one environment of a B747VecEnv (core/controller.py:43-360)."""

    def __init__(self, venv, i):
        self._v, self._i = venv, i
        eng = venv.engine
        if eng.cfg.export_signals and eng.dtype == E.F64:
            from .core.model import ModelView
            self.model = ModelView(eng, i)
        else:
            self.model = _FieldModel(eng, i)
        self.use_storage = bool(eng.cfg.record_capacity)
        self._vartheta_func = None
        self._h_func = None

    # configuration shared by the whole batch
    tk = property(lambda s: s._v.tk)
    sample_time = property(lambda s: s._v.sample_time)
    action_max = property(lambda s: s._v.action_max)
    vartheta_max = property(lambda s: s._v.vartheta_max)
    ctrl_type = property(lambda s: s._v.ctrl_type)
    ctrl_mode = property(lambda s: s._v.ctrl_mode)
    reset_ref_mode = property(lambda s: s._v.reset_ref_mode)
    disturbance_mode = property(lambda s: s._v.disturbance_mode)
    use_limiter = property(lambda s: s._v.use_limiter)

    @property
    def use_ctrl(self):
        return bool(int(self._v.engine.get("flags")[self._i]) & 4)

    # the reference of env i: assigning a constant function re-targets the running episode, as
    # `ctrl.vartheta_func = lambda _: vref` does (neural/callbacks.py:73)
    @property
    def vartheta_func(self):
        return self._vartheta_func

    @vartheta_func.setter
    def vartheta_func(self, f):
        from .core.controller import _const_value
        self._vartheta_func = f
        if f is not None:
            v = _const_value(f, "vartheta_func (vectorised env)", require=True)
            self._v._set_env_field("vref", self._i, v)

    @property
    def h_func(self):
        return self._h_func

    @h_func.setter
    def h_func(self, f):
        from .core.controller import _const_value
        self._h_func = f
        if f is not None:
            v = _const_value(f, "h_func (vectorised env)", require=True)
            self._v._set_env_field("href", self._i, v)

    @property
    def vartheta_ref(self):
        eng = self._v.engine
        if self.use_ctrl:
            return float(eng.get("sig_vzh")[self._i])
        return float(eng.get("vref")[self._i])

    @property
    def err_vartheta(self):
        return self.vartheta_ref - self.model.state_dict['vartheta']

    @property
    def err_h(self):
        return self.model.hzh - self.model.state_dict['y']

    @property
    def is_done(self):
        return self.model.time >= self.tk

    @property
    def storage(self):
        """Controller.storage of env i: the running episode as recorded after every model step
        (core/controller.py:209-228).  Needs B747VecEnv(record_capacity=...)."""
        eng = self._v.engine
        if not eng.cfg.record_capacity:
            return Storage()
        return Storage({k: list(v) for k, v in eng.recorder_read(self._i).items() if len(v)})

    def quality(self):
        """core/controller.py:334-336."""
        vr = self.vartheta_ref
        return math.exp(-60 * 0.1 * self.model.ITSE / (self.tk * vr ** 2))

    def stepinfo_SS(self, use_backup=False):
        return self._stepinfo("SS", 'vartheta', 'vartheta_ref', use_backup)

    def stepinfo_CS(self, use_backup=False):
        return self._stepinfo("CS", 'y', 'hzh', use_backup)

    def _stepinfo(self, which, sig, ref, finished):
        eng = self._v.engine
        if eng.cfg.track_transfer:  # the in-kernel tracker; use_backup = the most recently finished episode
            m = eng.transfer_metrics(which, finished=bool(finished))[self._i]
            val = lambda x: None if x != x else float(x)
            return {'overshoot': val(m[0]), 'static_error': val(m[3]), 'rise_time': val(m[1]), 'settling_time': val(m[2])}
        st = self.storage.storage
        if sig not in st or 't' not in st:
            raise ValueError('Вычисление хар-к ПП недоступно: ошибка хранилища.')
        return calc_stepinfo(st[sig], st[ref][-1], ts=st['t'])


class VecEnvItem:
    """ControllerEnv-shaped view of one environment of a B747VecEnv (env/ctrl_env.py:61-282): what SubprocVecEnv's
    get_attr / set_attr / env_method reach in a worker process."""

    def __init__(self, venv, i):
        self.__dict__["_v"] = venv
        self.__dict__["_i"] = i
        self.__dict__["ctrl"] = VecCtrlView(venv, i)

    observation_type = property(lambda s: s._v.observation_type)
    reward_type = property(lambda s: s._v.reward_type)
    norm_obs = property(lambda s: s._v.norm_obs)
    norm_act = property(lambda s: s._v.norm_act)
    observation_space = property(lambda s: s._v.observation_space)
    action_space = property(lambda s: s._v.action_space)
    reward_range = (0, 1)

    @property
    def state_box(self):
        """The observation env i returned last."""
        return np.array(self._v._last_obs_row(self._i), dtype=np.float64)

    def get_reward(self, action=None):
        return float(self._v._last_rew_row(self._i))

    def is_done(self):
        return self.ctrl.is_done

    def seed(self, seed=None):
        return [seed]

    def reset(self, state0=None):
        """ControllerEnv.reset of this environment alone: random draw (state0 None) or Controller.reset(state0) with
        the view's constant reference."""
        self._v._reset_env(self._i, state0, self.ctrl)
        return np.zeros(self._v.observation_space.shape)

    def __getattr__(self, name):  # anything else: the batch-wide attribute
        return getattr(self.__dict__["_v"], name)

    def __setattr__(self, name, value):
        if name in ("ctrl",):
            self.__dict__[name] = value
        else:
            setattr(self._v, name, value)


class B747VecEnv(_VecEnvBase):
    def __init__(self, num_envs, observation_type=ObservationType.PID_LIKE, reward_type=RewardType.CLASSIC,
                 norm_obs=True, norm_act=True, ctrl_type=CtrlType.MANUAL, ctrl_mode=CtrlMode.DIRECT_CONTROL,
                 reset_ref_mode=None, disturbance_mode=None, tk=20, sample_time=0.05, action_max=17 * np.pi / 180,
                 vartheta_max=10 * np.pi / 180, use_limiter=False, aero_err=None, reward_config=None, seed=1,
                 dtype=E.F32, device=0, device_tensors=False, env_id_offset=0, monitor=True, copy_outputs=True,
                 record_capacity=0, track_transfer=False, export_signals=False):
        from .core.controller import ResetRefMode
        if reset_ref_mode is None:
            reset_ref_mode = ResetRefMode.CONST  # a VecEnv auto-resets, which needs the random reset
        self.observation_type, self.reward_type = observation_type, reward_type
        self.norm_obs, self.norm_act = norm_obs, norm_act
        self.ctrl_type, self.ctrl_mode = ctrl_type, ctrl_mode
        self.reset_ref_mode, self.disturbance_mode, self.use_limiter = reset_ref_mode, disturbance_mode, use_limiter
        self.engine = E.BatchEngine(
            n_envs=num_envs, dtype=dtype, device=device, obs_type=_val(observation_type), rew_type=_val(reward_type),
            norm_obs=norm_obs, norm_act=norm_act, ctrl_type=_val(ctrl_type), ctrl_mode=_val(ctrl_mode, E.MODE_NONE),
            reset_ref_mode=_val(reset_ref_mode), disturbance_mode=_val(disturbance_mode, E.DIST_NONE),
            use_limiter=use_limiter, tk=tk, sample_time=sample_time, action_max=action_max, vartheta_max=vartheta_max,
            aero_err=aero_err, reward_config=reward_config, seed=seed, auto_reset=True, env_layer=True,
            env_id_offset=env_id_offset, record_capacity=record_capacity, track_transfer=track_transfer,
            export_signals=export_signals)
        self.num_envs = int(num_envs)
        self.observation_space, self.action_space = make_spaces(observation_type, norm_obs, norm_act, action_max)
        if _VecEnvBase is not object:
            _VecEnvBase.__init__(self, self.num_envs, self.observation_space, self.action_space)
        self.device_tensors = bool(device_tensors)
        self.monitor = bool(monitor)
        # copy_outputs=False: step_wait returns views of the pinned result buffers, which rotate between two sets --
        # an array stays valid until the step after the next one (SB3's collect_rollouts reads `_last_obs` once after
        # the following env.step); True (default) returns fresh arrays like SubprocVecEnv does
        self.copy_outputs = bool(copy_outputs)
        self.tk, self.sample_time, self.action_max, self.vartheta_max = tk, sample_time, action_max, vartheta_max
        self._t0 = time.time()
        self._actions = None
        self._seed = seed
        # SB3 wants one info dict per env and step; building 10^5..10^6 dicts per step would dominate the step, so the
        # empty ones are shared between steps and only the environments that finished get a fresh dict
        self._no_infos = [{} for _ in range(self.num_envs)]
        self._infos_list = list(self._no_infos)
        self._infos_dirty = []
        self._items = {}
        od = self.engine.obs_dim
        self._packed = (not self.device_tensors) and dtype == E.F32
        self._last = None  # (obs, rew) arrays of the last step
        self._keep = []
        if self.device_tensors:
            self._act_d, self._obs_d, self._rew_d, self._done_d, self._term_d = self.engine.alloc_io(terminal_obs=True)
        elif self._packed:
            self._act_h = self._pin((self.num_envs,), np.float32)
            self._out4 = [self._pin((self.num_envs, self.engine.record_floats), np.float32) for _ in range(2)]
            self._bits = self._pin(((self.num_envs + 31) // 32,), np.int32)  # one done bit per env
            self._flip = 0
        else:
            dt = self.engine.np_dtype
            self._act_h = self._pin((self.num_envs,), dt)
            self._obs = self._pin((self.num_envs, od), dt)
            self._rew = self._pin((self.num_envs,), dt)
            self._done = self._pin((self.num_envs,), np.uint8)
            self._term = self._pin((self.num_envs, od), dt)

    def _pin(self, shape, dtype):
        arr, owner = _pinned(shape, dtype)
        self._keep.append(owner)
        return arr

    # ---- VecEnv API ------------------------------------------------------------------------
    def reset(self):
        if self.device_tensors:
            self.engine.reset(self._obs_d)
            self.engine.synchronize()
            return self._obs_d
        self.engine.reset()
        self.engine.synchronize()
        # every exported signal is zero after initialize (env/ctrl_env.py:273-278)
        obs = np.zeros((self.num_envs, self.engine.obs_dim), self.engine.np_dtype)
        self._last = (obs, np.zeros(self.num_envs, self.engine.np_dtype))
        return obs

    def step_async(self, actions):
        self._actions = actions

    def step_wait(self):
        a = self._actions
        if self.device_tensors:
            self._act_d.copy_(a.reshape(self.num_envs))
            # run on the handle's stream after torch's current stream has produced the actions
            th = self.engine._th()
            th.cuda.current_stream().synchronize()
            self.engine.step(self._act_d, self._obs_d, self._rew_d, self._done_d, self._term_d)
            self.engine.synchronize()
            done_any = bool(self._done_d.any().item())
            infos = self._infos(self._done_d.cpu().numpy(), self._term_d) if done_any else self._clean_infos()
            self._last = (self._obs_d, self._rew_d)
            return self._obs_d, self._rew_d, self._done_d.bool(), infos
        np.copyto(self._act_h, np.asarray(a).reshape(self.num_envs), casting="unsafe")
        if self._packed:
            out = self._out4[self._flip]
            self._flip ^= 1
            self.engine.step_host_packed(self._act_h, out, self._bits)
            done = np.unpackbits(self._bits.view(np.uint8), bitorder="little")[:self.num_envs].view(bool)
            od = self.engine.obs_dim
            obs, rew = out[:, :od], out[:, od]
            if self.copy_outputs:
                obs, rew = obs.copy(), rew.copy()
            infos = self._clean_infos()
            if done.any():
                idx = np.flatnonzero(done)
                infos = self._infos_idx(idx, obs[idx].copy())   # the record holds the observation BEFORE the auto-reset
                obs[idx] = 0.0                                  # ... and the reset observation is all zeros
            self._last = (obs, rew)
            return obs, rew, done, infos
        self.engine.step_host(self._act_h, self._obs, self._rew, self._done, self._term)
        done = self._done.astype(bool)
        infos = self._infos(self._done, self._term) if done.any() else self._clean_infos()
        obs, rew = self._obs.copy(), self._rew.copy()
        self._last = (obs, rew)
        return obs, rew, done, infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def _clean_infos(self):
        for i in self._infos_dirty:
            self._infos_list[i] = self._no_infos[i]
        self._infos_dirty = []
        return self._infos_list

    def _infos(self, done, term):
        idx = np.nonzero(done)[0]
        if not len(idx):
            return self._clean_infos()
        dev = hasattr(term, "cpu")
        rows = term[idx] if not dev else term[th_index(term, idx)]
        return self._infos_idx(idx, rows)

    def _infos_idx(self, idx, rows):
        """One info dict per env (SB3's contract) at O(finished envs) per step: the list object is reused, the entries of
        the envs that finished in the PREVIOUS step go back to the shared empty dict, the ones that finished now get
        {"terminal_observation", "episode"}.  (SB3 consumes `infos` within the step that returned it.)"""
        infos = self._infos_list
        for i in self._infos_dirty:
            infos[i] = self._no_infos[i]
        idx_l = idx.tolist()
        dev = hasattr(rows, "cpu")
        rows_l = [r.clone() for r in rows] if dev else list(rows)
        if self.monitor:
            ret, ln = self.engine.last_episode_of(idx)   # only the finished envs' records
            t = round(time.time() - self._t0, 6)
            for i, row, r, l in zip(idx_l, rows_l, ret.tolist(), ln.tolist()):
                infos[i] = {"terminal_observation": row, "episode": {"r": r, "l": l, "t": t}}
        else:
            for i, row in zip(idx_l, rows_l):
                infos[i] = {"terminal_observation": row}
        self._infos_dirty = idx_l
        return infos

    def close(self):
        self.engine.close()

    def seed(self, seed=None):
        """SB3's env.seed(s) (neural/agent.py:80): re-keys the Philox stream of every later random reset; like
        SubprocVecEnv.seed the return value is one entry per env (env i is seeded with seed + i there; here the global
        env id is part of the Philox counter, so one key serves all)."""
        if seed is not None:
            self.engine.set_seed(int(seed))
            self._seed = int(seed)
        return [None if seed is None else int(seed) + i for i in range(self.num_envs)]

    # ---- per-environment views ----------------------------------------------------------------------------
    def _item(self, i):
        i = int(i)
        if not 0 <= i < self.num_envs:
            raise IndexError(i)
        it = self._items.get(i)
        if it is None:
            it = self._items[i] = VecEnvItem(self, i)
        return it

    class _Envs:
        def __init__(self, v):
            self._v = v

        def __len__(self):
            return self._v.num_envs

        def __getitem__(self, i):
            if isinstance(i, slice):
                return [self._v._item(k) for k in range(*i.indices(self._v.num_envs))]
            return self._v._item(i if i >= 0 else self._v.num_envs + i)

        def __iter__(self):
            return (self._v._item(i) for i in range(self._v.num_envs))

    @property
    def envs(self):
        return B747VecEnv._Envs(self)

    @property
    def ctrl(self):
        return self._item(0).ctrl

    def _indices(self, indices):
        if indices is None:
            return range(self.num_envs)
        if isinstance(indices, (int, np.integer)):
            return [int(indices)]
        return [int(i) for i in indices]

    def get_attr(self, attr_name, indices=None):
        return [getattr(self._item(i), attr_name) for i in self._indices(indices)]

    def set_attr(self, attr_name, value, indices=None):
        for i in self._indices(indices):
            setattr(self._item(i), attr_name, value)

    def env_method(self, method_name, *args, indices=None, **kwargs):
        return [getattr(self._item(i), method_name)(*args, **kwargs) for i in self._indices(indices)]

    def env_is_wrapped(self, wrapper_class, indices=None):
        return [False for _ in self._indices(indices)]

    def _set_env_field(self, name, i, value):
        v = self.engine.get(name)
        v[i] = float(value)
        self.engine.set(name, v)

    def _last_obs_row(self, i):
        if self._last is None:
            return np.zeros(self.engine.obs_dim)
        o = self._last[0][i]
        return o.cpu().numpy() if hasattr(o, "cpu") else o

    def _last_rew_row(self, i):
        if self._last is None:
            return 0.0
        r = self._last[1][i]
        return float(r.item()) if hasattr(r, "item") else float(r)

    def _reset_env(self, i, state0, ctrl):
        mask = np.zeros(self.num_envs, np.uint8)
        mask[i] = 1
        th = self.engine._th()
        m = th.from_numpy(mask).to(th.device("cuda", self.engine.cfg.device))
        if state0 is None:
            self.engine.reset(mask=m)
        else:
            from .core.controller import _const_value
            vref = _const_value(ctrl.vartheta_func, "vartheta_func", require=True) if ctrl.vartheta_func else 0.0
            href = _const_value(ctrl.h_func, "h_func", require=True) if ctrl.h_func else 11000.0
            eps = [E.episode(state0, vref=vref, h_ref=href, use_ctrl=ctrl.use_ctrl)] * self.num_envs
            self.engine.reset_to(eps, mask=m)
        self.engine.synchronize()

    def episode_stats(self):
        """(episodes, sum of returns, sum of lengths, sum of squared returns) since the last call."""
        return self.engine.episode_stats()

    # ---- checkpoint / resume ----------------------------------------------------------------------------
    def get_state(self):
        """Checkpoint of every env: {"engine": the handle's state blob (BatchEngine.save_state, a device tensor),
        "obs", "rew": copies of what the last reset or step returned (None before the first reset)}."""
        obs, rew = self._last if self._last is not None else (None, None)
        cp = lambda x: None if x is None else (x.clone() if hasattr(x, "clone") else np.array(x, copy=True))
        return {"engine": self.engine.save_state(), "obs": cp(obs), "rew": cp(rew)}

    def set_state(self, state):
        """Restore a get_state() checkpoint of an env created with the same arguments; returns the observation to
        continue from (SB3's `_last_obs`), as reset() would."""
        self.engine.load_state(state["engine"])
        self._clean_infos()
        od, dt = self.engine.obs_dim, self.engine.np_dtype
        obs, rew = state["obs"], state["rew"]
        if self.device_tensors:
            if obs is None:
                self._obs_d.zero_()
                self._rew_d.zero_()
            else:
                self._obs_d.copy_(obs)
                self._rew_d.copy_(rew)
            self._last = (self._obs_d, self._rew_d)
            return self._obs_d
        host = lambda x: np.array(x.cpu().numpy() if hasattr(x, "cpu") else x, dtype=dt, copy=True)
        obs = np.zeros((self.num_envs, od), dt) if obs is None else host(obs)
        rew = np.zeros(self.num_envs, dt) if rew is None else host(rew)
        self._last = (obs, rew)
        return obs.copy()

    @property
    def unwrapped(self):
        return self

    def render(self, mode="human"):
        pass
