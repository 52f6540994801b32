"""Kernel instantiations and branches that only a non-default Config or a large batch selects, against the CPU oracle
bit for bit: the 8-slot nearest-n list (Config.n > 4) and the masked 4-slot one (Config.n < 4), distance ties in the
nearest-n merge, step_n0_kernel's MINB = 8 build (no intruders, more than 2^18 envs), more than 128 intruders (flag
words outside registers) up to the 4096 cap, observation parameters changed between steps (Q12), and the device relabel
reward with Config.n != 4."""
import numpy as np
import pytest

from helpers import GOLDEN_VARIANTS, assert_state_equal, config_class
from test_nearest_ties import nearest_config, tie_states

pytestmark = pytest.mark.gpu


def _pair(vk, cfg_cls, N, B, mode, seed, auto_reset=True):
    from gca_b200 import variants
    from gca_b200.batched import BatchedAircraftEnv
    from oracle import oracle as orc
    env = BatchedAircraftEnv(GOLDEN_VARIANTS[vk], B, cfg_cls, n_intruders=N, mode=mode, draws="philox", seed=seed)
    ref = orc.OracleEnv(variants.make_config(GOLDEN_VARIANTS[vk], cfg_cls), B, N, draws=1, trig=orc.TRIG_SHARED,
                        seed=seed, f32_positions=mode == "fast", auto_reset=auto_reset)
    return env, ref


def _actions(env, rng, fast):
    import torch
    B = env.num_envs
    if env.continuous:
        a = rng.uniform(-1, 1, (B, 2))
        if fast:
            a = a.astype(np.float32).astype(np.float64)
        return a, torch.as_tensor(a, device=env.device).to(env.real)
    a = rng.randint(0, 3 if env.cfg.action_kind in (2, 3) else 9, B)
    return np.stack([a, np.zeros(B)], -1).astype(np.float64), torch.as_tensor(a.astype(np.int32), device=env.device)


def _same_outputs(env, ref, cast, what, rows=None):
    sel = (lambda x: x) if rows is None else (lambda x: x[rows])
    assert np.array_equal(sel(env.info.cpu().numpy()), sel(ref.info)), what
    assert np.array_equal(sel(env.done.cpu().numpy()), sel(ref.done)), what
    assert np.array_equal(sel(env.reward.cpu().numpy()), sel(cast(ref.reward))), what
    if env.obs_dim:
        assert np.array_equal(sel(env.obs.cpu().numpy()), sel(cast(ref.obs))), what
    if env.is_goal_env:
        assert np.array_equal(sel(env.achieved.cpu().numpy()), sel(cast(ref.achieved))), what
        assert np.array_equal(sel(env.desired.cpu().numpy()), sel(cast(ref.desired))), what
    if env.nearest is not None:
        assert np.array_equal(sel(env.nearest.cpu().numpy()), sel(cast(ref.nearest))), what


def rollout_vs_oracle(vk, cfg_cls, N, B, T, mode, seed, auto_reset=True, every_state=False):
    """Philox rollout with random actions; every output after every step and the whole state at the end bit for bit.
    Without auto-reset the finished envs are reset by mask."""
    fast = mode == "fast"
    env, ref = _pair(vk, cfg_cls, N, B, mode, seed, auto_reset)
    cast = (lambda x: x.astype(np.float32)) if fast else (lambda x: x)
    assert np.array_equal(env.reset().cpu().numpy(), cast(ref.reset()))
    rng = np.random.RandomState(seed + 1)
    events = np.zeros(6, np.int64)
    for t in range(T):
        a_host, a_dev = _actions(env, rng, fast)
        env.step(a_dev, auto_reset=auto_reset)
        ref.step(a_host)
        _same_outputs(env, ref, cast, (vk, N, mode, t))
        events += np.bincount(ref.info, minlength=6)
        if every_state:
            assert_state_equal(env.get_state(), ref.state, "state at step %d" % t, skip=())
        if not auto_reset and ref.done.any():
            done = ref.done.copy()
            env.reset(mask=done)
            ref.reset(mask=done)
            assert np.array_equal(env.obs.cpu().numpy(), cast(ref.obs)), t
    st = env.get_state()
    assert_state_equal(st, ref.state, "final state", skip=())
    assert np.array_equal(st["tick"], ref.state["tick"])
    env.close()
    return events


# ------------------------------------------------------------------------------------------------ nearest-n widths
NEAREST_CASES = [(vk, n, N) for vk in ("d9her", "d3her") for n in (1, 3, 5, 8) for N in sorted({n + 1, 33, 200})]


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("vk,n,N", NEAREST_CASES)
def test_nearest_widths_rollout_bit_exact_vs_oracle(vk, n, N, mode):
    """Config.n in {1, 3, 5, 8}: the 4-slot list masked to n, and the 8-slot list (write_obs_nearest<FAITH, 8>)."""
    B = 333 if N == 200 else 1000
    events = rollout_vs_oracle(vk, nearest_config(vk, n), N, B, 40, mode, seed=17 * n + N)
    assert events[0] > 0


@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_nearest_width8_masked_resets_vs_oracle(mode):
    events = rollout_vs_oracle("d9her", nearest_config("d9her", 8), 33, 777, 60, mode, seed=5, auto_reset=False)
    assert events[1] + events[2] > 0


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("n", [4, 8])
@pytest.mark.parametrize("vk", ["d9her", "d3her"])
def test_nearest_ties_on_device_vs_oracle(vk, n, mode):
    """Intruders at exactly equal distances (test_nearest_ties.tie_states): observe(), then one step - the nearest pass
    of a step runs behind the spawn phase - with the tied groups spread over the kernel's four sub-lanes."""
    fast = mode == "fast"
    B, N = 500, 40
    env, ref = _pair(vk, nearest_config(vk, n), N, B, mode, seed=3, auto_reset=True)
    cast = (lambda x: x.astype(np.float32)) if fast else (lambda x: x)
    st = tie_states(B, N, n, mixed=not fast, seed=7 * n + (not fast))
    env.set_state(st)
    for k, v in st.items():
        ref.state[k][...] = v
    assert np.array_equal(env.observe().cpu().numpy(), cast(ref.observe()))
    assert np.array_equal(env.achieved.cpu().numpy(), cast(ref.achieved))
    rng = np.random.RandomState(n)
    for t in range(2):
        a_host, a_dev = _actions(env, rng, fast)
        env.step(a_dev)
        ref.step(a_host)
        _same_outputs(env, ref, cast, (vk, n, mode, t))
    assert_state_equal(env.get_state(), ref.state, "after the steps", skip=())
    env.close()


# ------------------------------------------------------------------------------------------------ no intruders
@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("vk", ["env", "her", "dher"])
def test_n0_above_2p18_envs_vs_oracle(vk, mode):
    """N = 0 with B > 2^18 runs step_n0_kernel<FAITH, 8> (the MINB = 8 build)."""
    rollout_vs_oracle(vk, config_class(vk), 0, (1 << 18) + 37, 15, mode, seed=21)


def test_n0_at_2p18_envs_vs_oracle():
    """B = 2^18 exactly: the last batch size of the MINB = 1 build."""
    rollout_vs_oracle("env", config_class("env"), 0, 1 << 18, 6, "fast", seed=22)


def test_n0_bench_size_vs_oracle():
    """bench.py's 4 Mi-env N = 0 workload (FAST), a few steps."""
    rollout_vs_oracle("env", config_class("env"), 0, 4 * 1024 * 1024, 3, "fast", seed=23)


# ------------------------------------------------------------------------------------------------ wide intruder counts
@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("vk,N,B", [("her", 129, 300), ("d9her", 200, 300), ("d3her", 300, 200), ("mctsrnd", 150, 300)])
def test_more_than_128_intruders_vs_oracle(vk, N, B, mode):
    """Past N = 128 the flag words leave registers: own-first streaming kernel (her, word 5), nearest pass, d3her's
    shaped-nearest minimum, the random-intruder turn pass and drift (non-zero position_sigma)."""
    cfg = config_class(vk)
    if vk == "mctsrnd":
        cfg = type("CfgDrift", (cfg,), {"position_sigma": 0.3})
    rollout_vs_oracle(vk, cfg, N, B, 30, mode, seed=N + B)


@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_intruder_cap_4096_vs_oracle(mode):
    rollout_vs_oracle("env", config_class("env"), 4096, 40, 5, mode, seed=31, every_state=True)


# ------------------------------------------------------------------------------------------------ mid-run Config refresh
# (width, height, diagonal) between steps; 800 (the default) again at the end.  Every width here passes
# gca_div1_is_exact (so does every f32 significand sampled while writing this test): the FAST vector layout keeps the
# OM = 1 streaming kernel; the refresh must still re-derive the division constants of every kernel.
REFRESH = [(640, 480, 1000.0), (1024, 768, 1131.37), (500, 900, 777.7), (800, 800, 800.0)]


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("vk", ["env", "her", "d9her"])
def test_refresh_observation_params_mid_run_vs_oracle(vk, mode):
    fast = mode == "fast"
    cfg_cls = type("CfgMutable", (config_class(vk),), {})
    B, N = 600, 40
    env, ref = _pair(vk, cfg_cls, N, B, mode, seed=41)
    cast = (lambda x: x.astype(np.float32)) if fast else (lambda x: x)
    assert np.array_equal(env.reset().cpu().numpy(), cast(ref.reset()))
    rng = np.random.RandomState(42)
    for t in range(5 * len(REFRESH)):
        if t % 5 == 4:
            W, H, D = REFRESH[t // 5]
            cfg_cls.window_width, cfg_cls.window_height, cfg_cls.diagonal = W, H, D
            env.refresh_observation_params()
            ref.cfg.ob_window_width, ref.cfg.ob_window_height = float(W), float(H)
            if vk == "d9her":
                ref.cfg.ob_diagonal = float(D)
            assert env.cfg.ob_window_width == W and env.cfg.window_width == config_class(vk).window_width
        a_host, a_dev = _actions(env, rng, fast)
        env.step(a_dev)
        ref.step(a_host)
        _same_outputs(env, ref, cast, (vk, mode, t))
    assert_state_equal(env.get_state(), ref.state, "final state", skip=())
    env.close()


# ------------------------------------------------------------------------------------------------ input reward
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("n", [1, 8])
def test_input_reward_nearest_widths_vs_numpy(n, dtype):
    """gca_input_reward with Config.n in {1, 8} on 256 * 40 + 1 rows (a ragged last block)."""
    import torch
    from gca_b200 import replay
    from Simulators.config import Config
    from test_gpu_relabel import _input_reward_numpy
    c = type("CfgIR%d" % n, (Config,), {"n": n, "intruder_size": 8})
    m, dim = 256 * 40 + 1, 4 + 5 * n + 2
    rng = np.random.RandomState(n)
    x = rng.uniform(0.05, 0.95, (m, dim))
    near = rng.rand(m) < 0.5                                     # listed intruders and goals next to the ownship
    for j in range(n):
        x[near, 4 + 5 * j:6 + 5 * j] = x[near, 0:2] + rng.uniform(-0.03, 0.03, (int(near.sum()), 2))
    x[::3, -2:] = x[::3, 0:2] + rng.uniform(-0.02, 0.02, (len(x[::3]), 2))
    x = x.astype(dtype)
    r, d = replay.compute_input_reward(torch.as_tensor(x, device="cuda"), c)
    want = np.array([_input_reward_numpy(v, c) for v in x])
    assert np.array_equal(r.cpu().numpy(), want)
    assert np.array_equal(d.cpu().numpy(), ((want == 10) | (want == -10)).astype(np.uint8))
    kinds = set(np.select([want == c.NMAC_penalty, want == c.conflict_penalty, want == c.goal_reward], [1, 2, 3], 0).tolist())
    assert kinds == {0, 1, 2, 3}
