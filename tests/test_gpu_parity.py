"""GPU parity tests proper: the CUDA path (through the C ABI) against the reference goldens
and against the CPU oracle on the same inputs.

Bars (north star): conflict / NMAC / goal / done flags, conflict counters and draw counts
bit-exact; positions, headings, rewards and observations within 1e-9 relative of the numpy
reference in the faithful (fp64) mode.  Against the oracle evaluated with the shared
sincos/log (gca_math.h) everything is bit-exact, in both modes, at every size.
"""
import numpy as np
import pytest

from helpers import (FAST_TOL, GOAL_VARIANTS, GOLDEN_CASES, GOLDEN_N, GOLDEN_VARIANTS, STATE_KEYS, assert_state_equal, config_class,
                     fast_obs_tol, golden_actions, golden_config, golden_state, load_trace)

pytestmark = pytest.mark.gpu

RTOL = 1e-9     # fp64-mode tolerance of the north star (values); flags are compared exactly


def _torch():
    import torch
    return torch


def make_gpu(vk, n, B, mode, draws, seed=0):
    from gca_b200.batched import BatchedAircraftEnv
    return BatchedAircraftEnv(GOLDEN_VARIANTS[vk], B, config_class(vk), n_intruders=n, mode=mode, draws=draws, seed=seed)


def make_oracle(vk, n, B, draws, trig, seed=0, tape=None, f32=False, auto_reset=False):
    from oracle import oracle as orc
    return orc.OracleEnv(golden_config(vk), B, n, draws=draws, trig=trig, seed=seed, tape=tape, f32_positions=f32,
                         auto_reset=auto_reset)


def gpu_actions(env, a):
    torch = _torch()
    if env.continuous:
        return torch.as_tensor(np.ascontiguousarray(a[:, :2]), device=env.device).to(env.real)
    return torch.as_tensor(np.ascontiguousarray(a[:, 0]).astype(np.int32), device=env.device)


def close(a, b):
    return np.allclose(a, b, rtol=RTOL, atol=1e-300)


@pytest.mark.parametrize("vk,n", GOLDEN_CASES)
def test_golden_replay_faithful(vk, n):
    """Free-running replay of the reference traces: same start state, same actions, same draws."""
    torch = _torch()
    from oracle import oracle as orc
    g = load_trace(vk, n)
    B = g["tape"].shape[0]
    tape = np.nan_to_num(g["tape"], nan=0.0)
    env = make_gpu(vk, n, B, "faithful", "tape")
    ref = make_oracle(vk, n, B, 0, orc.TRIG_SHARED, tape=tape)       # bit-exact twin of the kernel
    her = vk in GOAL_VARIANTS

    # reset from the tape start
    D = env.obs_dim                                              # 0 for the image env: its vector observation is empty
    env.set_tape(tape)
    obs = env.reset().cpu().numpy()[:, :D]
    ref.reset()
    assert np.array_equal(env.tape_cursor.cpu().numpy(), np.broadcast_to(g["cur_reset0"], (B,)))
    assert_state_equal(env.get_state(), ref.state, "reset vs oracle %s n=%d" % (vk, n))
    assert np.array_equal(obs, ref.obs)
    plain = np.nonzero(g["kind_id"] == 0)[0]
    assert_state_equal(env.get_state(), golden_state(g, "s0_", plain), "reset vs reference", rows=plain,
                       skip=("ep_steps", "own_vel", "ivel"))
    assert close(obs[plain], g["obs0"][plain])

    # engineered start states
    st = golden_state(g, "s0_")
    env.set_state(st)
    for k, v in st.items():
        ref.state[k][...] = v
    assert close(env.observe().cpu().numpy()[:, :D], g["obs0"])

    acts = golden_actions(vk, g)
    exact = total = 0
    for t in range(acts.shape[1]):
        what = "%s n=%d step %d" % (vk, n, t)
        obs, rew, done, info = env.step(gpu_actions(env, acts[:, t]), auto_reset=False)
        ref.step(acts[:, t])
        obs, rew, done, info = obs.cpu().numpy()[:, :D], rew.cpu().numpy(), done.cpu().numpy(), info.cpu().numpy()
        # --- against the reference itself
        assert np.array_equal(info, g["event"][:, t]), what
        assert np.array_equal(done, g["done"][:, t]), what
        assert np.array_equal(env.tape_cursor.cpu().numpy(), g["cur_after"][:, t]), what
        assert close(rew, g["reward"][:, t]), what
        assert close(obs, g["obs"][:, t]), what
        if her:
            assert close(env.achieved.cpu().numpy(), g["ag"][:, t]) and close(env.desired.cpu().numpy(), g["dg"][:, t])
        if vk == "d3her":
            assert close(env.nearest.cpu().numpy(), g["nearest"][:, t]), what
            assert np.array_equal(env.nearest.cpu().numpy(), ref.nearest), what
        state = env.get_state()
        want = golden_state(g, "sa_", (slice(None), t))
        assert np.array_equal(state["no_conflict"], want["no_conflict"]), what
        assert np.array_equal(state["iflag"], want["iflag"]), what
        assert np.array_equal(state["ipos_is_f64"], want["ipos_is_f64"]), what
        for k in ("own_pos", "own_hs", "ipos", "ivel", "goal"):
            assert close(state[k], want[k]), (what, k)
        exact += int(np.array_equal(obs, g["obs"][:, t])) + int(np.array_equal(state["own_pos"], want["own_pos"]))
        total += 2
        # --- against the oracle twin: every bit
        assert np.array_equal(obs, ref.obs) and np.array_equal(rew, ref.reward), what
        assert_state_equal(state, ref.state, what + " vs oracle", skip=())
        if done.any():
            env.reset(mask=done)
            ref.reset(mask=done)
            rows = np.nonzero(done)[0]
            assert close(env.obs.cpu().numpy()[rows, :D], g["reset_obs"][rows, t]), what
            assert np.array_equal(env.obs.cpu().numpy()[rows, :D], ref.obs[rows]), what
        assert np.array_equal(env.tape_cursor.cpu().numpy(), g["cur_after_reset"][:, t]), what
    env.close()
    print("%s n=%d: %d/%d step outputs bit-identical to the reference" % (vk, n, exact, total))


@pytest.mark.parametrize("vk,n", GOLDEN_CASES)
def test_golden_replay_fast(vk, n):
    """The fp32 ("fast") mode - what bench.py measures - against the traces recorded from the unmodified reference:
    free-running replay from the recorded start state with the recorded draws.  Flags, done, conflict counters,
    per-intruder conflict flags and the number of draws consumed must be IDENTICAL over the whole horizon; positions,
    observations, rewards inside the stated fp32 tolerance (helpers.FAST_TOL; DESIGN.md section 2).  And every bit
    equals the oracle's f32_positions twin evaluated with the shared sincos / log."""
    from oracle import oracle as orc
    g = load_trace(vk, n)
    B = g["tape"].shape[0]
    tape = np.nan_to_num(g["tape"], nan=0.0)
    env = make_gpu(vk, n, B, "fast", "tape")
    ref = make_oracle(vk, n, B, 0, orc.TRIG_SHARED, tape=tape, f32=True)
    D = env.obs_dim
    st = golden_state(g, "s0_")
    st["ipos"] = st["ipos"].astype(np.float32).astype(np.float64)   # the fast mode's storage rule (a retried spawn's f64
    st["ipos_is_f64"][...] = 0                                      # position is kept rounded to f32: Q3 dropped)
    env.set_state(st)
    env.set_tape(tape, cursor=np.broadcast_to(g["cur_reset0"], (B,)))
    for k, v in st.items():
        ref.state[k][...] = v
    ref.cursor[...] = g["cur_reset0"]
    f64 = lambda x: x.cpu().numpy().astype(np.float64)
    otol = fast_obs_tol(vk)
    assert np.abs(f64(env.observe())[:, :D] - g["obs0"]).max(initial=0) <= otol
    acts = golden_actions(vk, g)
    if env.continuous:                         # the fast mode takes its actions as f32 (a VecEnv action buffer)
        acts = acts.astype(np.float32).astype(np.float64)
    worst = {"pos": 0.0, "obs": 0.0, "reward": 0.0}
    for t in range(acts.shape[1]):
        what = "%s n=%d step %d" % (vk, n, t)
        obs, rew, done, info = env.step(gpu_actions(env, acts[:, t]), auto_reset=False)
        ref.step(acts[:, t])
        done, info = done.cpu().numpy(), info.cpu().numpy()
        # --- against the reference itself: exact flags and draw counts
        assert np.array_equal(info, g["event"][:, t]) and np.array_equal(done, g["done"][:, t]), what
        assert np.array_equal(env.tape_cursor.cpu().numpy(), g["cur_after"][:, t]), what
        state = env.get_state()
        want = golden_state(g, "sa_", (slice(None), t))
        assert np.array_equal(state["no_conflict"], want["no_conflict"]) and np.array_equal(state["iflag"], want["iflag"]), what
        # --- values inside the stated tolerance
        dp = max(np.abs(state["own_pos"] - want["own_pos"]).max(), np.abs(state["ipos"] - want["ipos"]).max(initial=0))
        do = np.abs(f64(obs)[:, :D] - g["obs"][:, t]).max(initial=0)
        dr = np.abs(f64(rew) - g["reward"][:, t]).max()
        assert dp <= FAST_TOL["pos"] and do <= otol and dr <= FAST_TOL["reward"], (what, dp, do, dr)
        worst = {"pos": max(worst["pos"], dp), "obs": max(worst["obs"], do), "reward": max(worst["reward"], dr)}
        if vk in GOAL_VARIANTS:
            gtol = FAST_TOL["pos"] if vk == "dher" else FAST_TOL["obs"]
            assert np.abs(f64(env.achieved) - g["ag"][:, t]).max() <= gtol and np.abs(f64(env.desired) - g["dg"][:, t]).max() <= gtol
        if vk == "d3her":
            assert np.abs(f64(env.nearest) - g["nearest"][:, t]).max() <= FAST_TOL["nearest"], what
        # --- against the oracle twin: every bit
        assert np.array_equal(obs.cpu().numpy()[:, :D], ref.obs.astype(np.float32)), what
        assert np.array_equal(rew.cpu().numpy(), ref.reward.astype(np.float32)), what
        assert_state_equal(state, ref.state, what + " vs oracle", skip=())
        if done.any():
            env.reset(mask=done)
            ref.reset(mask=done)
            rows = np.nonzero(done)[0]
            assert np.abs(f64(env.obs)[rows, :D] - g["reset_obs"][rows, t]).max(initial=0) <= otol, what
        assert np.array_equal(env.tape_cursor.cpu().numpy(), g["cur_after_reset"][:, t]), what
    env.close()
    print("%s n=%d fast mode: max |d| positions %.2e px, observation %.2e, reward %.2e" % (vk, n, worst["pos"], worst["obs"], worst["reward"]))


@pytest.mark.parametrize("vk,n", [("env", 80), ("env2", 80), ("her", 3), ("dher", 80), ("mcts", 80), ("d9her", 80),
                                  ("d9her", 12), ("d3her", 80), ("mctsrnd", 80), ("mctsrnd", 3), ("stack", 80), ("stack", 3)])
def test_teacher_forced_single_steps(vk, n):
    """Load each recorded reference state, take ONE step, compare with the next recorded state
    (chaotic divergence cannot hide a bug)."""
    g = load_trace(vk, n)
    B, T = g["actions"].shape[:2]
    tape = np.nan_to_num(g["tape"], nan=0.0)
    env = make_gpu(vk, n, B, "faithful", "tape")
    acts = golden_actions(vk, g)
    for t in range(1, T):
        ok = g["done"][:, t - 1] == 0                       # a finished env was reset in between
        env.set_state(golden_state(g, "sa_", (slice(None), t - 1)))
        env.set_tape(tape, cursor=g["cur_before"][:, t])
        obs, rew, done, info = env.step(gpu_actions(env, acts[:, t]), auto_reset=False)
        assert np.array_equal(info.cpu().numpy()[ok], g["event"][ok, t])
        assert np.array_equal(done.cpu().numpy()[ok], g["done"][ok, t])
        assert close(rew.cpu().numpy()[ok], g["reward"][ok, t])
        assert close(obs.cpu().numpy()[ok][:, :env.obs_dim], g["obs"][ok, t])
        st = env.get_state()
        want = golden_state(g, "sa_", (slice(None), t))
        assert np.array_equal(st["no_conflict"][ok], want["no_conflict"][ok])
        assert np.array_equal(st["iflag"][ok], want["iflag"][ok])
        assert close(st["ipos"][ok], want["ipos"][ok]) and close(st["own_pos"][ok], want["own_pos"][ok])
    env.close()


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("vk,n,B,T", [("env", 80, 4096, 40), ("env2", 80, 2048, 40), ("her", 33, 1000, 40),
                                      ("dher", 3, 1000, 60), ("mcts", 80, 1024, 40), ("env", 0, 5000, 30),
                                      ("env", 1, 777, 60), ("env2", 200, 300, 30), ("d9her", 80, 2048, 60),
                                      ("d9her", 5, 999, 80), ("d9her", 33, 500, 40), ("d3her", 80, 2048, 60),
                                      ("d3her", 7, 640, 80), ("mctsrnd", 80, 2048, 60), ("mctsrnd", 7, 700, 80),
                                      ("mctsrnd", 1, 333, 60)])
def test_philox_rollout_bit_exact_vs_oracle(vk, n, B, T, mode):
    """On-device Philox draws, VecEnv auto-reset: every output and the whole state must equal the
    CPU oracle driven by the same counter-based stream - bit for bit (ragged batch sizes included)."""
    from oracle import oracle as orc
    fast = mode == "fast"
    env = make_gpu(vk, n, B, mode, "philox", seed=1234)
    ref = make_oracle(vk, n, B, 1, orc.TRIG_SHARED, seed=1234, f32=fast, auto_reset=True)
    cast = (lambda x: x.astype(np.float32)) if fast else (lambda x: x)
    assert np.array_equal(env.reset().cpu().numpy(), cast(ref.reset()))
    rng = np.random.RandomState(5)
    events = np.zeros(6, np.int64)
    for t in range(T):
        if env.continuous:
            a = rng.uniform(-1, 1, (B, 2))
            if fast:
                a = a.astype(np.float32).astype(np.float64)
        else:
            a = np.stack([rng.randint(0, 3 if vk in ("dher", "d3her") else 9, B), np.zeros(B)], -1).astype(np.float64)
        obs, rew, done, info = env.step(gpu_actions(env, a))
        ref.step(a)
        info = info.cpu().numpy()
        assert np.array_equal(info, ref.info), t
        assert np.array_equal(done.cpu().numpy(), ref.done), t
        assert np.array_equal(rew.cpu().numpy(), cast(ref.reward)), t
        assert np.array_equal(obs.cpu().numpy(), cast(ref.obs)), t
        if env.is_goal_env:
            assert np.array_equal(env.achieved.cpu().numpy(), cast(ref.achieved))
            assert np.array_equal(env.desired.cpu().numpy(), cast(ref.desired))
        if env.nearest is not None:
            assert np.array_equal(env.nearest.cpu().numpy(), cast(ref.nearest)), t
        events += np.bincount(info, minlength=6)
    assert_state_equal(env.get_state(), ref.state, "final state", skip=())
    assert np.array_equal(env.get_state()["tick"], ref.state["tick"])
    env.close()
    print(vk, n, mode, "events", events.tolist())


def test_full_size_bit_exact_vs_oracle():
    """BASELINE.json size: 65,536 envs x 80 intruders, fast mode, continuous actions."""
    from oracle import oracle as orc
    vk, n, B, T = "env2", 80, 65536, 12
    env = make_gpu(vk, n, B, "fast", "philox", seed=99)
    ref = make_oracle(vk, n, B, 1, orc.TRIG_SHARED, seed=99, f32=True, auto_reset=True)
    assert np.array_equal(env.reset().cpu().numpy(), ref.reset().astype(np.float32))
    rng = np.random.RandomState(11)
    for t in range(T):
        a = rng.uniform(-1, 1, (B, 2)).astype(np.float32).astype(np.float64)
        obs, rew, done, info = env.step(gpu_actions(env, a))
        ref.step(a)
        assert np.array_equal(info.cpu().numpy(), ref.info) and np.array_equal(done.cpu().numpy(), ref.done)
        assert np.array_equal(obs.cpu().numpy(), ref.obs.astype(np.float32))
        assert np.array_equal(rew.cpu().numpy(), ref.reward.astype(np.float32))
    assert_state_equal(env.get_state(), ref.state, "final state", skip=())
    env.close()


def test_step_host_equals_device_path():
    torch = _torch()
    a_env = make_gpu("env", 80, 2048, "fast", "philox", seed=3)
    b_env = make_gpu("env", 80, 2048, "fast", "philox", seed=3)
    o1 = a_env.reset().cpu().numpy()
    o2 = b_env.reset_host()
    assert np.array_equal(o1, o2)
    rng = np.random.RandomState(0)
    for _ in range(10):
        a = rng.randint(0, 9, 2048).astype(np.int32)
        o, r, d, i = a_env.step(torch.as_tensor(a, device="cuda"))
        ho, hr, hd, hi = b_env.step_host(a)
        assert np.array_equal(o.cpu().numpy(), ho) and np.array_equal(r.cpu().numpy(), hr)
        assert np.array_equal(d.cpu().numpy(), hd) and np.array_equal(i.cpu().numpy(), hi)
    h2d, d2h = b_env.host_io_bytes()
    assert h2d == 2048 * 4 and d2h == 2048 * (328 * 4 + 4 + 1 + 1)


@pytest.mark.parametrize("vk", ["env", "mctsrnd"])
def test_state_roundtrip_and_independence_of_batch_split(vk):
    """set_state(get_state()) is the identity, and env b evolves the same whatever batch it sits in
    (Philox is keyed by the global env id: the basis of multi-GPU sharding, SURVEY 8(e))."""
    from gca_b200.batched import BatchedAircraftEnv
    torch = _torch()
    cfgc = config_class(vk)
    name = GOLDEN_VARIANTS[vk]
    whole = BatchedAircraftEnv(name, 600, cfgc, n_intruders=40, seed=5)
    part = BatchedAircraftEnv(name, 200, cfgc, n_intruders=40, seed=5, env_id0=400)
    whole.reset(); part.reset()
    rng = np.random.RandomState(1)
    for _ in range(25):
        a = torch.as_tensor(rng.randint(0, 9, 600).astype(np.int32), device="cuda")
        whole.step(a); part.step(a[400:].contiguous())
    sw, sp = whole.get_state(), part.get_state()
    for k in STATE_KEYS:
        assert np.array_equal(sw[k][400:], sp[k]), k
    clone = BatchedAircraftEnv(name, 600, cfgc, n_intruders=40, seed=5)
    clone.set_state(sw)
    a = torch.as_tensor(rng.randint(0, 9, 600).astype(np.int32), device="cuda")
    o1 = whole.step(a)[0].cpu().numpy()
    o2 = clone.step(a)[0].cpu().numpy()
    assert np.array_equal(o1, o2)


def test_compute_reward_matches_reference():
    import os
    from helpers import GOLDEN
    from gca_b200 import abi
    from gca_b200.batched import compute_reward
    torch = _torch()
    g = np.load(os.path.join(GOLDEN, "her_reward.npz"))
    dev = lambda x: torch.as_tensor(x, device="cuda")
    r = compute_reward(dev(g["ag_n"]), dev(g["g_n"]), 20.0, abi.OBS_HER).cpu().numpy()
    assert np.array_equal(r, g["r_her"]) and np.all(np.signbit(r))          # always -0.0 (Q14)
    assert np.array_equal(compute_reward(dev(g["ag_p"]), dev(g["g_p"]), 20.0, abi.OBS_DHER).cpu().numpy(), g["r_dher"])
    assert np.array_equal(compute_reward(dev(g["ag_p"]), dev(g["g_p"]), 20.0, abi.OBS_HER).cpu().numpy(), g["r_her_pix"])
    # f32 inputs (what a VecEnv buffer holds) keep the whole norm in f32, like numpy
    from oracle import oracle as orc
    ag32, g32 = g["ag_p"].astype(np.float32), g["g_p"].astype(np.float32)
    want = orc.compute_reward(ag32, g32, 20.0, abi.OBS_DHER)
    assert np.array_equal(compute_reward(dev(ag32), dev(g32), 20.0, abi.OBS_DHER).cpu().numpy(), want)
    # a relabel batch of BASELINE config #3: M = 4 * 65,536 pairs
    rng = np.random.RandomState(0)
    ag = rng.uniform(0, 800, (4 * 65536, 2)); gg = ag + rng.uniform(-30, 30, ag.shape)
    assert np.array_equal(compute_reward(dev(ag), dev(gg), 20.0, abi.OBS_DHER).cpu().numpy(),
                          orc.compute_reward(ag, gg, 20.0, abi.OBS_DHER))
    # the same relabel without the k copies of the achieved goals (gca_compute_reward_tiled): [B, 2] against [k, B, 2]
    agb = ag[:65536]
    gk = (agb[None] + rng.uniform(-30, 30, (4, 65536, 2)))
    got = compute_reward(dev(agb), dev(gk), 20.0, abi.OBS_DHER).cpu().numpy()
    assert got.shape == (4, 65536)
    assert np.array_equal(got, orc.compute_reward(np.broadcast_to(agb, gk.shape).reshape(-1, 2), gk.reshape(-1, 2), 20.0,
                                                  abi.OBS_DHER).reshape(4, 65536))


@pytest.mark.parametrize("vk", ["env2", "mctsrnd"])
@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_long_rollout_with_explicit_masked_resets_vs_oracle(mode, vk):
    """No auto-reset: a finished env keeps its terminal state (after an NMAC the intruders behind the hit one
    must sit where they were, Q9) until the caller resets exactly those envs.  After the first masked reset the
    envs of one tile no longer agree on which position plane is current; 250 steps with random actions reach
    every event kind many times.  Everything is compared with the oracle, bit for bit, after every step."""
    from oracle import oracle as orc
    n, B, T = 80, 1536, 250 if vk == "env2" else 120
    fast = mode == "fast"
    env = make_gpu(vk, n, B, mode, "philox", seed=77)
    ref = make_oracle(vk, n, B, 1, orc.TRIG_SHARED, seed=77, f32=fast, auto_reset=False)
    cast = (lambda x: x.astype(np.float32)) if fast else (lambda x: x)
    assert np.array_equal(env.reset().cpu().numpy(), cast(ref.reset()))
    rng = np.random.RandomState(9)
    events = np.zeros(6, np.int64)
    resets = 0
    for t in range(T):
        if env.continuous:
            a = rng.uniform(-1, 1, (B, 2))
            if fast:
                a = a.astype(np.float32).astype(np.float64)
        else:
            a = np.stack([rng.randint(0, 9, B), np.zeros(B)], -1).astype(np.float64)
        obs, rew, done, info = env.step(gpu_actions(env, a), auto_reset=False)
        ref.step(a)
        done = done.cpu().numpy()
        info = info.cpu().numpy()
        assert np.array_equal(info, ref.info) and np.array_equal(done, ref.done), t
        assert np.array_equal(rew.cpu().numpy(), cast(ref.reward)), t
        assert np.array_equal(obs.cpu().numpy(), cast(ref.obs)), t
        events += np.bincount(info, minlength=6)
        if t % 10 == 9 or t == T - 1:
            assert_state_equal(env.get_state(), ref.state, "state at step %d" % t, skip=())
        if done.any():
            resets += int(done.sum())
            o = env.reset(mask=done).cpu().numpy()
            ref.reset(mask=done)
            assert np.array_equal(o, cast(ref.obs)), t
    assert events[1] > 0 and events[2] > 0 and (events[4] > 0 or vk != "env2") and resets > 0, events    # NMAC, conflict, wall all happened
    env.close()
    print(mode, "events", events.tolist(), "resets", resets)


def test_kernels_per_step_and_profile():
    """gca_step_launches / gca_profile_*: what bench.py uses for gpu_launches and for the roofline of the
    dominant kernel."""
    torch = _torch()
    env = make_gpu("env", 80, 4096, "fast", "philox", seed=1)
    assert env.kernels_per_step == 2                      # ownship role + streaming pass; finish + spawn phase
    env.reset()
    a = torch.zeros(4096, dtype=torch.int32, device="cuda")
    env.profile(True)
    for _ in range(5):
        env.step(a)
    p = env.read_profile()
    env.profile(False)
    assert p["steps"] == 5 and p["intruders_ms"] > 0 and p["finish_ms"] > 0 and p["own_ms"] >= 0 and p["spawn_ms"] >= 0
    env.step(a)
    assert env.read_profile()["steps"] == 0
    env.close()
    e0 = make_gpu("env", 0, 64, "fast", "philox", seed=1)
    assert e0.kernels_per_step == 1                       # no intruders: one kernel (ownship + finish, thread = env)
    e0.close()
    g = load_trace("env", 3)
    et = make_gpu("env", 3, g["tape"].shape[0], "faithful", "tape")
    assert et.kernels_per_step == 3                       # tape replay respawns in place: no spawn kernel
    et.close()
    er = make_gpu("mctsrnd", 80, 64, "fast", "philox", seed=1)
    assert er.kernels_per_step == 3                       # + the turn / six-entry observation pass
    er.close()


@pytest.mark.parametrize("case", range(10))
def test_random_configurations_bit_exact_vs_oracle(case):
    """Non-default parameters (window, radii, speeds, noise, intruder count, batch size drawn at random per case; the
    constant-division fast paths do not all qualify then): kernels and oracle must still agree on every bit."""
    from gca_b200 import variants
    from gca_b200.batched import BatchedAircraftEnv
    from oracle import oracle as orc
    rng = np.random.RandomState(1000 + case)
    vk = ["env", "env2", "her", "dher", "mcts", "d9her", "d3her", "env2", "mctsrnd", "mctsrnd"][case]
    base = config_class(vk)
    W, H = [(800, 800), (640, 480), (1024, 768), (500, 900)][rng.randint(4)]
    over = dict(window_width=W, window_height=H, diagonal=float(rng.choice([800, 1000, 1131.37])),
                minimum_separation=float(rng.uniform(10, 30)), NMAC_dist=float(rng.uniform(2, 8)),
                initial_min_dist=float(rng.uniform(40, 120)), goal_radius=float(rng.uniform(10, 40)),
                min_speed=float(rng.uniform(1.0, 2.0)), max_speed=float(rng.uniform(2.2, 3.5)),
                d_speed=float(rng.uniform(0.05, 0.3)), speed_sigma=float(rng.uniform(0.0, 0.1)),
                d_heading=float(rng.uniform(0.02, 0.2)), heading_sigma=float(rng.uniform(0.0, 0.1)))
    if vk == "mctsrnd":                     # the per-step drift of the random-intruder env (a separate stream: cases 0-7 keep their draws)
        over["position_sigma"] = float(np.random.RandomState(5000 + case).choice([0.0, 0.25, -0.4]))
    cfg_cls = type("Cfg%d" % case, (base,), over)
    n = int(rng.randint(6, 100))
    B = int(rng.randint(100, 700))
    mode = "fast" if case % 2 == 0 else "faithful"
    fast = mode == "fast"
    cfg = variants.make_config(GOLDEN_VARIANTS[vk], cfg_cls)
    env = BatchedAircraftEnv(GOLDEN_VARIANTS[vk], B, cfg_cls, n_intruders=n, mode=mode, draws="philox", seed=77 + case)
    ref = orc.OracleEnv(cfg, B, n, draws=1, trig=orc.TRIG_SHARED, seed=77 + case, f32_positions=fast, auto_reset=True)
    cast = (lambda x: x.astype(np.float32)) if fast else (lambda x: x)
    assert np.array_equal(env.reset().cpu().numpy(), cast(ref.reset()))
    for t in range(40):
        if env.continuous:
            a = rng.uniform(-1, 1, (B, 2))
            if fast:
                a = a.astype(np.float32).astype(np.float64)
        else:
            a = np.stack([rng.randint(0, 3 if vk in ("dher", "d3her") else 9, B), np.zeros(B)], -1).astype(np.float64)
        obs, rew, done, info = env.step(gpu_actions(env, a))
        ref.step(a)
        assert np.array_equal(info.cpu().numpy(), ref.info), (vk, t)
        assert np.array_equal(done.cpu().numpy(), ref.done), (vk, t)
        assert np.array_equal(rew.cpu().numpy(), cast(ref.reward)), (vk, t)
        assert np.array_equal(obs.cpu().numpy(), cast(ref.obs)), (vk, t)
    assert_state_equal(env.get_state(), ref.state, "final state", skip=())
    env.close()
    print(vk, mode, "W,H", W, H, "N", n, "B", B)


def test_host_path_async_equals_device_path():
    """gca_step_host_begin / _wait (two steps in flight, double-buffered downloads) return, step for step, what the
    device-resident path returns for the same seed and actions; mixing in the synchronous gca_step_host keeps the order."""
    import torch
    B, n, T = 777, 20, 24
    a = make_gpu("env2", n, B, "fast", "philox", seed=31)
    b = make_gpu("env2", n, B, "fast", "philox", seed=31)
    assert np.array_equal(a.reset().cpu().numpy(), b.reset_host())
    rng = np.random.RandomState(2)
    acts = [rng.uniform(-1, 1, (B, 2)).astype(np.float32) for _ in range(T)]
    want = []
    for t in range(T):
        o, r, d, i = a.step(torch.as_tensor(acts[t], device="cuda"))
        want.append((o.cpu().numpy().copy(), r.cpu().numpy().copy(), d.cpu().numpy().copy(), i.cpu().numpy().copy()))

    def same(got, t):
        for x, y in zip(got, want[t]):
            assert np.array_equal(np.asarray(x), y), t
    b.step_host_begin(acts[0])
    for t in range(1, 10):                       # pipelined: step t is begun before step t - 1 is waited for
        b.step_host_begin(acts[t])
        same(b.step_host_wait(), t - 1)
    same(b.step_host_wait(), 9)
    for t in range(10, 14):                      # synchronous calls in between
        same(b.step_host(acts[t]), t)
    b.step_host_begin(acts[14])
    b.step_host_begin(acts[15])
    with pytest.raises(Exception):
        b.step_host_begin(acts[16])              # a third step in flight is refused
    same(b.step_host_wait(), 14)
    same(b.step_host_wait(), 15)
    for t in range(16, T):
        b.step_host_begin(acts[t])
        same(b.step_host_wait(), t)
    a.close()
    b.close()
