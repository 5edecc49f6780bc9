"""Host-side logic: tick thresholds, substep count, Philox, reward constants, sharding and the
world_size-2 episode-statistics reduction (gloo)."""
import ctypes
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_done_tick_is_float64_exact(oracle):
    from b747_rl_ctrl_b200 import _lib
    L = _lib.load()
    for tk in [20, 20.0, 3.0, 0.05, 0.07, 0.3, 1e-9, 59.99, 60, 0.29, 0.57, 1.13, 7.0, 12.34]:
        n = _lib.done_tick_of(tk)
        assert n * 0.01 >= tk and (n == 0 or (n - 1) * 0.01 < tk)
        assert L.b747_done_tick(float(tk)) == n
        assert oracle.olib().b747o_done_tick(float(tk)) == n
        assert oracle.done_tick_of(tk) == n
    assert _lib.done_tick_of(20) == 2000
    assert _lib.done_tick_of(0.0) == 0


def test_substeps_follow_python_round():
    from b747_rl_ctrl_b200 import _lib
    assert _lib.substeps_of(None) == 1
    assert _lib.substeps_of(0.05) == 5 and _lib.substeps_of(0.1) == 10 and _lib.substeps_of(0.01) == 1
    assert _lib.substeps_of(0.025) == 2      # round(2.5) -> 2 (banker's), like core/controller.py:261
    assert _lib.substeps_of(0.035) == round(0.035 / 0.01)
    # the reference's loop `round(round(t/dt) % round(Ts/dt)) != 0` ends after exactly K steps from tick 0
    for st in (0.01, 0.02, 0.05, 0.1):
        K = _lib.substeps_of(st)
        tick, n = 0, 0
        while True:
            tick += 1; n += 1
            if round(round((tick * 0.01) / 0.01) % round(st / 0.01)) == 0:
                break
        assert n == K


def test_philox_known_answers(oracle):
    from b747_rl_ctrl_b200 import _lib
    L = _lib.load()
    kats = [([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
            ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
            ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
             [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])]
    for ctr, key, exp in kats:
        for fn in (L.b747_philox4x32, oracle.olib().b747o_philox4x32):
            c = (ctypes.c_uint32 * 4)(*ctr); k = (ctypes.c_uint32 * 2)(*key); o = (ctypes.c_uint32 * 4)()
            fn(c, k, o)
            assert list(o) == exp


def test_reset_distributions(oracle):
    """Controller.reset's distributions (core/controller.py:148-165) from the Philox stream."""
    O = oracle
    cfg = O.make_cfg(seed=3)
    eps = [O.draw_episode(cfg, i, 0) for i in range(4000)]
    s0 = np.array([list(e.state0) for e in eps])
    assert (s0[:, 0] == 0).all() and (s0[:, 4] == 0).all()
    assert 1000 <= s0[:, 1].min() and s0[:, 1].max() <= 11000 and abs(s0[:, 1].mean() - 6000) < 150
    assert 100 <= s0[:, 2].min() and s0[:, 2].max() <= 265
    assert -20 <= s0[:, 3].min() and s0[:, 3].max() <= 20
    assert np.abs(s0[:, 5]).max() <= 1e-3
    v = np.array([e.vref_const for e in eps])
    assert (np.abs(v) >= math.pi / 180 - 1e-15).all() and (np.abs(v) <= 10 * math.pi / 180).all()
    assert 0.45 < (v > 0).mean() < 0.55
    # streams depend on (seed, env, episode) only
    a, b = O.draw_episode(cfg, 17, 5), O.draw_episode(cfg, 17, 5)
    assert list(a.state0) == list(b.state0) and a.vref_const == b.vref_const
    assert list(O.draw_episode(cfg, 17, 6).state0) != list(a.state0)
    cfg_o = O.make_cfg(seed=3, reset_ref_mode=O.RESET_OSCILLATING)
    e = O.draw_episode(cfg_o, 1, 0)
    assert e.oscillating == 1 and sum(e.osc_A) <= 10 * math.pi / 180 + 1e-12 and all(0.01 <= f <= 0.5 for f in e.osc_f)


def test_reward_constants_match_reference_formulae():
    from b747_rl_ctrl_b200 import _lib
    k = _lib.reward_constants(0)
    assert k[:3] == [2 / 5, 2 / 5, 1 / 5] and k[3] == 2 and k[4] == 0.3 and k[5] == 0.1
    assert k[6] == -math.log(0.8) / 10 and k[7] == -math.log(0.75) / 0.15   # calc_exp_k, tools/general.py:32-33
    k = _lib.reward_constants(0, {"k1": 1, "k2": 1, "k3": 2, "k0": 3})
    assert k[:4] == [0.25, 0.25, 0.5, 3]


def test_shard_ranges_cover_everything():
    from b747_rl_ctrl_b200.sharding import shard_range, summarize
    for n, g in [(8 * 2 ** 20, 8), (1000, 3), (7, 8), (65536, 4)]:
        spans = [shard_range(n, g, r) for r in range(g)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(spans[i][1] == spans[i + 1][0] for i in range(g - 1))
    s = summarize([4, 10.0, 1600, 30.0])
    assert s["ep_rew_mean"] == 2.5 and s["ep_len_mean"] == 400 and s["ep_rew_std"] == pytest.approx(math.sqrt(7.5 - 6.25))


def _stats_worker(rank, world, port, q):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from b747_rl_ctrl_b200.sharding import reduce_episode_stats, shard_range
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lo, hi = shard_range(1000, world, rank)
    # every rank contributes the statistics of its own env range
    local = np.array([hi - lo, float(sum(range(lo, hi))), 400.0 * (hi - lo), float(sum(i * i for i in range(lo, hi)))])
    out = reduce_episode_stats(local)
    dist.barrier()
    dist.destroy_process_group()
    q.put((rank, out.tolist()))


def test_stats_reduction_world_size_2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    ps = [ctx.Process(target=_stats_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = dict(q.get(timeout=120) for _ in ps)
    for p in ps:
        p.join(60)
        assert p.exitcode == 0
    exp = [1000.0, float(sum(range(1000))), 400000.0, float(sum(i * i for i in range(1000)))]
    assert res[0] == exp and res[1] == exp


def test_bench_reference_arm_prints_one_json_line():
    """bench.py --impl reference: ONE JSON line on stdout with the contract's keys (the CUDA arm shares the printer)."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1


@pytest.mark.gpu
def test_bench_dump_outputs_repeat_exactly(tmp_path):
    """bench.py --dump-outputs: obs / reward / done of the last timed step, identical from run to run."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for run in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--config", "fp64_4096", "--steps", "7",
                            "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / run)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout)["steps"] == 7
        dumps.append({n: np.load(tmp_path / run / f"{n}.npy") for n in ("obs", "reward", "done")})
    a, b = dumps
    assert a["obs"].shape == (4096, 3) and a["reward"].shape == a["done"].shape == (4096,)
    assert all(x.dtype == np.float64 for x in a.values())
    assert np.isfinite(a["obs"]).all() and set(np.unique(a["done"])) <= {0.0, 1.0}
    for n in a:
        assert np.array_equal(a[n], b[n]), n
