"""BatchEngine -- thin Python view of one b747_handle (one GPU, N environments resident in HBM).

Every number is produced by the sm_100a kernels behind libb747_b200.so; this module only marshals
pointers.  torch is used for device buffers and streams, nothing else.
"""
import ctypes
import math

import numpy as np

from . import _lib
from ._lib import F32, F64, B747Error, Cfg, Episode, check

# enum values == the reference's (core/controller.py:14-36, env/ctrl_env.py:16-30)
CTRL_FULL_AUTO, CTRL_AUTO, CTRL_SEMI_MANUAL, CTRL_MANUAL = 0, 1, 2, 3
MODE_DIRECT, MODE_ADD_PROC, MODE_ANG_VEL, MODE_ADD_DIRECT = 0, 1, 2, 3
MODE_NONE = -1  # ctrl_mode=None (CtrlType.AUTO / FULL_AUTO): action law as DIRECT, no rf reward term
RESET_NONE, RESET_CONST, RESET_OSCILLATING, RESET_HYBRID = -1, 0, 1, 2
DIST_NONE, DIST_AERO = -1, 0
OBS_PID_LIKE, OBS_SPEED_MODE, OBS_PID_AERO, OBS_PID_SPEED_AERO, OBS_MODEL_STATE = 0, 1, 2, 3, 4
REW_CLASSIC, REW_PID_LIKE, REW_QUALITY, REW_MINIMAL, REW_TF_REFERENCE = 0, 1, 2, 3, 4
OBS_DIM = {0: 3, 1: 5, 2: 8, 3: 10, 4: 7}
# per-env model tunables (b747_set_env_param) and their component counts, in the order of their Philox draw indices
ENV_PARAMS = {"m0": 1, "Iz": 1, "P": 1, "S": 1, "c_": 1, "PID_SS": 4, "PID_CS": 4}
ENV_PARAM_DRAW0 = 32


def make_cfg(n_envs, dtype=F32, device=0, obs_type=OBS_PID_LIKE, rew_type=REW_CLASSIC, ctrl_type=CTRL_MANUAL,
             ctrl_mode=MODE_DIRECT, reset_ref_mode=RESET_CONST, disturbance_mode=DIST_NONE, norm_obs=True,
             norm_act=True, use_limiter=False, tk=20.0, sample_time=0.05, action_max=17 * math.pi / 180,
             vartheta_max=10 * math.pi / 180, reward_config=None, aero_err=None, seed=1, auto_reset=True,
             env_layer=True, env_id_offset=0, export_signals=False, track_transfer=False, record_capacity=0):
    """Defaults are the canonical configuration main.py:88-121 trains (SURVEY.md 8d)."""
    c = Cfg()
    c.abi_version = _lib.ABI_VERSION
    c.device, c.dtype, c.n_envs = int(device), int(dtype), int(n_envs)
    c.obs_type, c.rew_type, c.ctrl_type, c.ctrl_mode = int(obs_type), int(rew_type), int(ctrl_type), int(ctrl_mode)
    c.reset_ref_mode, c.disturbance_mode = int(reset_ref_mode), int(disturbance_mode)
    c.norm_obs, c.norm_act, c.use_limiter = int(bool(norm_obs)), int(bool(norm_act)), int(bool(use_limiter))
    c.substeps = _lib.substeps_of(sample_time)
    c.auto_reset, c.env_layer = int(bool(auto_reset)), int(bool(env_layer))
    c.done_tick = _lib.done_tick_of(tk)
    c.env_id_offset, c.seed = int(env_id_offset), int(seed)
    c.tk, c.action_max, c.vartheta_max = float(tk), float(action_max), float(vartheta_max)
    c.sample_time = float(sample_time if sample_time else 0.01)
    for i, x in enumerate(_lib.reward_constants(rew_type, reward_config)):
        c.rew[i] = x
    if aero_err is not None:
        c.has_fixed_aero_err = 1
        for i in range(5):
            c.fixed_aero_err[i] = float(aero_err[i])
    c.export_signals = int(bool(export_signals))
    c.track_transfer = int(bool(track_transfer))
    c.record_capacity = int(record_capacity)
    return c


def episode(state0, vref=0.0, h_ref=11000.0, use_ctrl=False, osc=None, aero_err=None):
    e = Episode()
    for i in range(6):
        e.state0[i] = float(state0[i])
    e.vref_const, e.h_ref, e.use_ctrl = float(vref), float(h_ref), int(use_ctrl)
    if osc is not None:
        e.oscillating = 1
        for i in range(3):
            e.osc_A[i], e.osc_f[i] = float(osc[0][i]), float(osc[1][i])
    if aero_err is not None:
        for i in range(5):
            e.aero_err[i] = float(aero_err[i])
    return e


def _ptr(x):
    """Raw pointer of a torch tensor / numpy array / None."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return ctypes.c_void_p(x.ctypes.data)
    return ctypes.c_void_p(x.data_ptr())


class BatchEngine:
    """N environments on one GPU behind the C ABI."""

    def __init__(self, cfg=None, **kw):
        self._L = _lib.load()
        self.cfg = cfg if cfg is not None else make_cfg(**kw)
        self.n_envs = self.cfg.n_envs
        self.obs_dim = OBS_DIM[self.cfg.obs_type]
        self.dtype = self.cfg.dtype
        self.np_dtype = np.float64 if self.dtype == F64 else np.float32
        h = ctypes.c_void_p()
        check(self._L.b747_create(ctypes.byref(self.cfg), ctypes.byref(h)))
        self._h = h
        self._torch = None

    # -- lifecycle -----------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._L.b747_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream_ptr(self):
        return self._L.b747_stream(self._h)

    def use_stream(self, cuda_stream_ptr):
        check(self._L.b747_set_stream(self._h, ctypes.c_void_p(cuda_stream_ptr)))

    def synchronize(self):
        check(self._L.b747_synchronize(self._h))

    @property
    def launch_count(self):
        return int(self._L.b747_launch_count(self._h))

    # -- torch buffers (device memory plumbing) --------------------------------------
    def _th(self):
        if self._torch is None:
            import torch
            self._torch = torch
        return self._torch

    def torch_dtype(self):
        th = self._th()
        return th.float64 if self.dtype == F64 else th.float32

    def alloc_io(self, terminal_obs=False):
        """Device tensors (actions, obs, rew, done[, terminal_obs]) of the handle dtype."""
        th = self._th()
        dev = th.device("cuda", self.cfg.device)
        dt = self.torch_dtype()
        bufs = [th.zeros(self.n_envs, dtype=dt, device=dev), th.zeros(self.n_envs, self.obs_dim, dtype=dt, device=dev),
                th.zeros(self.n_envs, dtype=dt, device=dev), th.zeros(self.n_envs, dtype=th.uint8, device=dev)]
        if terminal_obs:
            bufs.append(th.zeros(self.n_envs, self.obs_dim, dtype=dt, device=dev))
        return bufs

    # -- reset / step ---------------------------------------------------------------------
    def reset(self, obs=None, mask=None):
        check(self._L.b747_reset(self._h, _ptr(mask), _ptr(obs)))

    def reset_to(self, episodes, obs=None, mask=None):
        """Explicit episodes (Controller.reset(state0)); mask: device uint8 tensor selecting the envs to reset."""
        arr = (Episode * self.n_envs)(*episodes)
        check(self._L.b747_reset_to_masked(self._h, arr, _ptr(mask), _ptr(obs)))

    def step(self, actions, obs, rew, done, terminal_obs=None):
        """Device pointers in, asynchronous on the handle's stream."""
        check(self._L.b747_step(self._h, _ptr(actions), _ptr(obs), _ptr(rew), _ptr(done), _ptr(terminal_obs)))

    def step_host(self, actions, obs=None, rew=None, done=None, terminal_obs=None):
        """Host (numpy) buffers: H2D actions, step, D2H results; returns (obs, rew, done[, terminal_obs])."""
        a = np.ascontiguousarray(np.asarray(actions, dtype=self.np_dtype).reshape(self.n_envs))
        obs = np.empty((self.n_envs, self.obs_dim), self.np_dtype) if obs is None else obs
        rew = np.empty(self.n_envs, self.np_dtype) if rew is None else rew
        done = np.empty(self.n_envs, np.uint8) if done is None else done
        check(self._L.b747_step_host(self._h, _ptr(a), _ptr(obs), _ptr(rew), _ptr(done), _ptr(terminal_obs)))
        if terminal_obs is not None:
            return obs, rew, done, terminal_obs
        return obs, rew, done

    @property
    def record_floats(self):
        """Floats per packed record: 4 * ceil((obs_dim + 1) / 4) -- obs, reward, zero padding."""
        return int(self._L.b747_packed_record_floats(self.cfg.obs_type))

    def step_packed(self, actions, out4, done_bits):
        """Device tensors: out4 [n_envs, record_floats] float32 = (obs before auto-reset, reward, padding), done_bits
        [(n_envs+31)//32] int32/uint32 (one bit per env).  f32 handles.  Asynchronous."""
        check(self._L.b747_step_packed(self._h, _ptr(actions), _ptr(out4), _ptr(done_bits)))

    def step_host_packed(self, actions, out4, done_bits):
        """Host buffers (float32 [n_envs], float32 [n_envs, record_floats], uint32 [(n_envs+31)//32]); page-locked buffers are read
        and written by the kernel directly (zero-copy).  Synchronised on return."""
        check(self._L.b747_step_host_packed(self._h, _ptr(actions), _ptr(out4), _ptr(done_bits)))

    def set_host_mode(self, mode):
        """step_host_packed with pinned buffers: -1 automatic, 0 staged copies, 1 zero-copy records, 2 zero-copy both."""
        check(self._L.b747_set_host_mode(self._h, int(mode)))

    def set_seed(self, seed):
        """env.seed(s): re-key the Philox stream of every later random reset."""
        check(self._L.b747_set_seed(self._h, int(seed) & (2 ** 64 - 1)))
        self.cfg.seed = int(seed) & (2 ** 64 - 1)

    def set_host_chunks(self, n_chunks):
        """Chunks of the copy/compute pipeline of step_host and of step_host_packed's staged copies (mode 0, pinned
        buffers): 0 = automatic, 1 = one launch."""
        check(self._L.b747_set_host_chunks(self._h, int(n_chunks)))

    def model_step(self, n_steps=1):
        check(self._L.b747_model_step(self._h, int(n_steps)))

    def model_initialize(self):
        check(self._L.b747_model_initialize(self._h))

    # -- named fields / params ----------------------------------------------------------------
    def field_names(self):
        return [self._L.b747_field_name(i).decode() for i in range(self._L.b747_n_fields())]

    def get(self, name):
        idx = self._L.b747_field_index(name.encode())
        if idx < 0:
            raise KeyError(name)
        out = np.empty(self.n_envs, np.float64)
        check(self._L.b747_get_field(self._h, idx, _ptr(out)))
        return out

    def set(self, name, values):
        idx = self._L.b747_field_index(name.encode())
        if idx < 0:
            raise KeyError(name)
        v = np.ascontiguousarray(np.broadcast_to(np.asarray(values, np.float64), (self.n_envs,)))
        check(self._L.b747_set_field(self._h, idx, _ptr(v)))

    def set_param(self, name, value):
        v = np.atleast_1d(np.asarray(value, np.float64))
        check(self._L.b747_set_param(self._h, name.encode(), v.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), len(v)))

    def get_param(self, name, n=1):
        v = np.zeros(n, np.float64)
        check(self._L.b747_get_param(self._h, name.encode(), v.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), n))
        return v if n > 1 else float(v[0])

    # -- trace: step-response metrics and the Storage recorder -------------------------------------------------
    METRIC_NAMES = ("overshoot", "rise_time", "settling_time", "static_error", "quality")

    def transfer_metrics(self, which="SS", finished=True):
        """calc_stepinfo (tools/general.py:46-61) + Controller.quality per env, computed in-kernel; [n_envs, 5] float64
        in METRIC_NAMES order, NaN where the reference returns None.  which: "SS" pitch / "CS" altitude."""
        out = np.empty((self.n_envs, 5), np.float64)
        check(self._L.b747_transfer_metrics(self._h, 0 if which == "SS" else 1, int(bool(finished)), _ptr(out)))
        return out

    def recorder_fields(self):
        return [self._L.b747_recorder_field_name(i).decode() for i in range(self._L.b747_recorder_n_fields())]

    def recorder_read(self, env=0):
        """The running episode of one env as {name: float64 array}, one entry per MODEL step (the reference's
        Storage after Controller._post_step, core/controller.py:209-228)."""
        names = self.recorder_fields()
        cap = self.cfg.record_capacity
        buf = np.zeros((len(names), max(cap, 1)), np.float64)
        n = ctypes.c_int32(0)
        check(self._L.b747_recorder_read(self._h, int(env), _ptr(buf), ctypes.byref(n)))
        return {nm: buf[k, :n.value].copy() for k, nm in enumerate(names)}

    # -- state save / load (checkpoint, resume, fork) --------------------------------------------------------
    def state_bytes(self, n=None):
        """Bytes of a state blob holding n envs (default: all) of this handle's configuration."""
        b = int(self._L.b747_state_bytes(ctypes.byref(self.cfg), self.n_envs if n is None else int(n)))
        if b < 0:
            check(b)
        return b

    def _device(self):
        return self._th().device("cuda", self.cfg.device)

    def _dev_index(self, idx):
        """Contiguous int32 device tensor of an index list (numpy array, sequence or tensor); None stays None."""
        if idx is None:
            return None
        th = self._th()
        t = idx if isinstance(idx, th.Tensor) else th.from_numpy(np.ascontiguousarray(idx, np.int32).reshape(-1))
        return t.to(device=self._device(), dtype=th.int32).contiguous().reshape(-1)

    def _order(self, after_torch):
        """after_torch: the handle's stream waits for what torch's current stream queued so far (index and blob
        tensors); else torch's current stream waits for the handle's."""
        th = self._th()
        dev = self._device()
        handle = th.cuda.ExternalStream(self.stream_ptr or 0, device=dev)
        cur = th.cuda.current_stream(dev)
        src, dst = (cur, handle) if after_torch else (handle, cur)
        ev = th.cuda.Event()
        ev.record(src)
        dst.wait_event(ev)

    def save_state(self, indices=None, out=None):
        """State blob (torch.uint8 device tensor) of the envs `indices` (numpy array or int32 device tensor; default
        every env in order): entry k holds env indices[k].  `out`: a preallocated uint8 device tensor of at least
        state_bytes(n) bytes.  Asynchronous; torch's current stream is ordered after the copy.  A checkpoint on disk
        is the blob's .cpu() copy."""
        th = self._th()
        idx = self._dev_index(indices)
        n = self.n_envs if idx is None else idx.numel()
        nb = self.state_bytes(n)
        if out is None:
            out = th.empty(nb, dtype=th.uint8, device=self._device())
        elif (out.dtype != th.uint8 or out.device != self._device() or not out.is_contiguous() or out.numel() < nb
              or out.data_ptr() % 16):
            raise ValueError(f"out must be a contiguous, 16-byte aligned uint8 tensor of at least {nb} bytes on "
                             f"{self._device()}")
        self._order(after_torch=True)
        check(self._L.b747_save_state(self._h, _ptr(idx), n, _ptr(out)))
        self._order(after_torch=False)
        return out

    def load_state(self, blob, indices=None, blob_indices=None):
        """Env indices[k] <- blob entry blob_indices[k] (either None: the identity; both None: every env from the entry
        of the same number).  blob: what save_state returned, on this device, another one or the host (copied here,
        and to a fresh tensor where it does not start 16-byte aligned).  Raises B747Error if the blob is not a state
        blob of this handle's dtype and configuration, ValueError if it is shorter than its header says.
        Synchronised."""
        th = self._th()
        b = blob if isinstance(blob, th.Tensor) else th.from_numpy(np.ascontiguousarray(blob).reshape(-1).view(np.uint8))
        if b.dtype != th.uint8 or b.dim() != 1:
            raise ValueError("blob must be a 1-D uint8 tensor (BatchEngine.save_state)")
        if b.numel() < 64:
            raise B747Error("not a state blob: shorter than its 64-byte header")
        head = b[:64].cpu().numpy()
        # magic, version, dtype (bytes 0-11) and configuration key (24-31) against a 0-env blob of this handle, so that a
        # foreign blob is refused like the C call refuses it before its size is judged by this handle's layout
        own = th.empty(64, dtype=th.uint8, device=self._device())
        self._order(after_torch=True)
        check(self._L.b747_save_state(self._h, None, 0, _ptr(own)))
        self._order(after_torch=False)
        own = own.cpu().numpy()
        if not (np.array_equal(head[:12], own[:12]) and np.array_equal(head[24:32], own[24:32])):
            raise B747Error("not a state blob of this handle's dtype and configuration (magic, version, dtype or key "
                            "differ)")
        n_blob = int(head[12:16].view(np.int32)[0])
        if n_blob < 0 or b.numel() < self.state_bytes(n_blob):
            raise ValueError(f"blob is shorter than a blob of its {n_blob} entries: truncated")
        b = b.to(self._device()).contiguous()
        if b.data_ptr() % 16:
            b = b.clone()   # fresh allocations are aligned
        idx, bidx = self._dev_index(indices), self._dev_index(blob_indices)
        if idx is not None and bidx is not None and idx.numel() != bidx.numel():
            raise ValueError("indices and blob_indices differ in length")
        n = idx.numel() if idx is not None else (bidx.numel() if bidx is not None else self.n_envs)
        self._order(after_torch=True)
        check(self._L.b747_load_state(self._h, _ptr(b), _ptr(bidx), _ptr(idx), n))

    # -- per-env model tunables (domain randomisation, gain sweeps) -------------------------------------------
    def _env_param_n(self, name):
        if name not in ENV_PARAMS:
            raise KeyError(f"not a per-env parameter: {name} (one of {', '.join(ENV_PARAMS)})")
        return ENV_PARAMS[name]

    def set_env_param(self, name, values, indices=None):
        """Env indices[k] (default: env k) takes values[k] ([n] or [n, 4] for PID_SS / PID_CS; numpy or a device
        tensor).  The first call puts the handle in per-env mode for good, every env starting from the whole-batch
        values.  Asynchronous, ordered after torch's current stream."""
        th = self._th()
        nc = self._env_param_n(name)
        v = values if isinstance(values, th.Tensor) else th.from_numpy(np.ascontiguousarray(values, np.float64))
        v = v.to(device=self._device(), dtype=th.float64).contiguous().reshape(-1)
        idx = self._dev_index(indices)
        n = v.numel() // nc
        if v.numel() != n * nc or (idx is not None and idx.numel() != n):
            raise ValueError(f"{name}: values must be [n] or [n, {nc}] with one row per index")
        self._order(after_torch=True)
        check(self._L.b747_set_env_param(self._h, name.encode(), _ptr(v), _ptr(idx), n))
        self._order(after_torch=False)

    def get_env_param(self, name, indices=None):
        """float64 device tensor of env indices[k]'s values (default: every env), [n] or [n, 4]; the whole-batch
        value for every env while the handle is not in per-env mode."""
        th = self._th()
        nc = self._env_param_n(name)
        idx = self._dev_index(indices)
        n = self.n_envs if idx is None else idx.numel()
        out = th.full((n, nc) if nc > 1 else (n,), float("nan"), dtype=th.float64, device=self._device())
        self._order(after_torch=True)
        check(self._L.b747_get_env_param(self._h, name.encode(), _ptr(idx), n, _ptr(out)))
        self._order(after_torch=False)
        return out

    def set_env_param_range(self, name, lo, hi):
        """From now on every random reset (b747_reset and the in-kernel auto-reset) draws each component of `name`
        uniformly in [lo, hi].  Enters per-env mode."""
        nc = self._env_param_n(name)
        lo = np.ascontiguousarray(np.broadcast_to(np.asarray(lo, np.float64), (nc,)))
        hi = np.ascontiguousarray(np.broadcast_to(np.asarray(hi, np.float64), (nc,)))
        dp = ctypes.POINTER(ctypes.c_double)
        check(self._L.b747_set_env_param_range(self._h, name.encode(), lo.ctypes.data_as(dp), hi.ctypes.data_as(dp), nc))

    def clear_env_param_range(self, name):
        """`name` keeps each env's current value through later resets."""
        check(self._L.b747_set_env_param_range(self._h, name.encode(), None, None, self._env_param_n(name)))

    # -- episode statistics ---------------------------------------------------------------------
    def episode_stats(self):
        """(episodes finished, sum of returns, sum of lengths, sum of squared returns) since the last call."""
        out = (ctypes.c_double * 4)()
        check(self._L.b747_episode_stats(self._h, out))
        return np.array(out)

    def last_episode_of(self, idx):
        """(return, length) of the most recently finished episode of the envs `idx` (VecMonitor's record of a step)."""
        idx = np.ascontiguousarray(idx, np.int32)
        ret = np.empty(len(idx), np.float64)
        ln = np.empty(len(idx), np.int32)
        check(self._L.b747_last_episode_of(self._h, _ptr(idx), len(idx), _ptr(ret), _ptr(ln)))
        return ret, ln

    def last_episode(self):
        ret = np.empty(self.n_envs, np.float64)
        ln = np.empty(self.n_envs, np.int32)
        check(self._L.b747_last_episode(self._h, _ptr(ret), _ptr(ln)))
        return ret, ln
