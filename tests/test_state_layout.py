"""Size of a state blob (b747_state_bytes) against the row-table formula of DESIGN.md §3.1, without a GPU.

A blob is a 64-byte header and then, for every per-env row the handle allocates, the n saved envs' entries padded to
16 bytes.  The row counts below are written out from the layout (b747_kernels_f32.cu: 14 double2 and 5 float4 groups;
b747_common.cuh: the float64 slots + six state0 rows, 2 x 9 tracker rows in `trk` and in `snap`, 13 recorder fields
per recorded model step); the library's field table supplies the slot and signal counts.
"""
import ctypes

import pytest

N_D_GROUPS, N_F_GROUPS, N_TRK = 14, 5, 9
SIZES = (1, 2, 77, (1 << 18) + 77)


@pytest.fixture(scope="module")
def L():
    from b747_rl_ctrl_b200 import _lib, build
    build.build_native()
    return _lib.load()


def _counts(L):
    names = [L.b747_field_name(i).decode() for i in range(L.b747_n_fields())]
    n_slot = names.index("state0_x")      # the float64 slots, state0_x..state0_wz, the exported signals, "tick", ...
    n_sig = names.index("tick") - (n_slot + 6)
    return n_slot, n_sig, L.b747_recorder_n_fields()


def _formula(L, dtype, n, signals, tracker, rec_cap):
    from b747_rl_ctrl_b200 import _lib
    n_slot, n_sig, n_rec = _counts(L)
    pad = lambda elem: (n * elem + 15) // 16 * 16
    if dtype == _lib.F32:
        rows = [(16, N_D_GROUPS), (16, N_F_GROUPS), (8, 1), (4, 1)] + ([(4, n_sig)] if signals else [])
    else:   # slots + state0, tick, flags, ep_idx, last_ret, last_len
        rows = [(8, n_slot + 6), (4, 1), (4, 1), (4, 1), (8, 1), (4, 1)] + ([(8, n_sig)] if signals else [])
    if tracker:
        rows += [(8, 2 * N_TRK), (8, 2 * N_TRK)]
    if rec_cap:
        rows += [(8, rec_cap * n_rec)]
    return 64 + sum(r * pad(e) for e, r in rows)


@pytest.mark.parametrize("dtype", ["f32", "f64"])
@pytest.mark.parametrize("extras", [False, True], ids=["plain", "signals-tracker-recorder"])
def test_state_bytes_equals_row_table(L, dtype, extras):
    from b747_rl_ctrl_b200 import _lib, engine
    dt = _lib.F32 if dtype == "f32" else _lib.F64
    kw = dict(export_signals=True, track_transfer=True, record_capacity=50) if extras else {}
    for n in SIZES:
        cfg = engine.make_cfg(n_envs=max(n, 4), dtype=dt, **kw)
        want = _formula(L, dt, n, extras, extras, 50 if extras else 0)
        assert L.b747_state_bytes(ctypes.byref(cfg), n) == want, (dtype, extras, n)


def test_canonical_f32_is_316_bytes_per_env(L):
    from b747_rl_ctrl_b200 import engine
    cfg = engine.make_cfg(n_envs=1 << 20)
    assert L.b747_state_bytes(ctypes.byref(cfg), 1 << 20) == 64 + 316 * (1 << 20)   # 14*16 + 5*16 + 8 + 4
    assert L.b747_state_bytes(ctypes.byref(cfg), 0) == 64


def test_state_bytes_ignores_what_a_blob_does_not_depend_on(L):
    from b747_rl_ctrl_b200 import engine
    a = engine.make_cfg(n_envs=100, seed=1, env_id_offset=0, record_capacity=7)
    b = engine.make_cfg(n_envs=5000, seed=9, env_id_offset=12345, device=3, record_capacity=7)
    assert L.b747_state_bytes(ctypes.byref(a), 100) == L.b747_state_bytes(ctypes.byref(b), 100)


def test_state_bytes_rejects_bad_arguments(L):
    from b747_rl_ctrl_b200 import _lib, engine
    cfg = engine.make_cfg(n_envs=4)
    assert L.b747_state_bytes(ctypes.byref(cfg), -1) == _lib.ERR_ARG
    assert L.b747_state_bytes(None, 4) == _lib.ERR_ARG
    cfg.dtype = 7
    assert L.b747_state_bytes(ctypes.byref(cfg), 4) == _lib.ERR_ARG
