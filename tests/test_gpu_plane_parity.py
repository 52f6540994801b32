"""Batches whose envs disagree on the current position plane, and Philox ticks past 2^31, stepped with auto-reset -
against the CPU oracle, bit for bit.

An env's tick (counters.z) addresses its Philox draws, and `tick & 1` picks which of the two position planes is current:
a step reads that plane and writes the other.  A masked reset advances the ticks of the reset envs only, and
gca_set_state takes any uint32 tick, so neighbouring envs - of one 32-env tile, of one aligned 8-env group, of one
128-byte line of a plane - can be on different planes.  Two things in the step depend on that:
- the FAST streaming pass discards (discard.global.L2) the lines of the plane it has just read when auto-reset is on;
  a line holds the positions of 8 envs, so it is only dead when all of its real envs read that plane;
- the spawn phase runs the respawns that finish_tile queued per env, keyed by the env's tick, which may be any uint32
  and wraps at 2^32.
"""
import numpy as np
import pytest

from helpers import GOLDEN_CASES, assert_state_equal, config_class, golden_actions, golden_state, load_trace
from test_gpu_config_paths import _actions, _pair, _same_outputs
from test_gpu_parity import gpu_actions, make_gpu, make_oracle

pytestmark = pytest.mark.gpu

NMAC, CONFLICT, GOAL, WALL = 1, 2, 3, 4
MODES = ["fast", "faithful"]


def mixed_groups(ticks, B, width):
    """Aligned groups of `width` envs (8: one 128-byte line of a FAST plane; 32: a tile) whose real envs hold both tick
    parities.  The padding lanes of a ragged last group do not count."""
    par = np.full(-(-B // width) * width, -1, np.int8)
    par[:B] = np.asarray(ticks, np.uint32)[:B] & 1
    g = par.reshape(-1, width)
    return int(np.count_nonzero((g == 0).any(1) & (g == 1).any(1)))


def _cast(mode):
    return (lambda x: x.astype(np.float32)) if mode == "fast" else (lambda x: x)


def _same_state(env, ref, what):
    st = env.get_state()
    assert_state_equal(st, ref.state, what, skip=())
    assert np.array_equal(st["tick"], ref.state["tick"]), what


def _set_both(env, ref, st):
    env.set_state(st)
    for k, v in st.items():
        ref.state[k][...] = v


def _masked_reset(env, ref, mask, cast, what):
    m = np.asarray(mask, np.uint8)
    o = env.reset(mask=m).cpu().numpy()
    ref.reset(mask=m)
    assert np.array_equal(o[:, :ref.D], cast(ref.obs)), what       # (D = 0: the image env has no vector observation)


# ------------------------------------------------------------------------------------------------ masked resets
ROLLOUT_CASES = [(vk, 80) for vk in ("env", "env2", "her", "dher", "mcts", "d9her", "d3her", "mctsrnd")] + \
                [("env2", n) for n in (0, 8, 33, 200)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("vk,N", ROLLOUT_CASES)
def test_masked_resets_then_auto_reset_steps_vs_oracle(vk, N, mode):
    """10 steps without auto-reset (finished envs reset by mask, plus one forced masked reset that leaves aligned 8-env
    groups on both planes), 40 auto-reset steps, then 20 more with a masked reset of a random subset every 5th step.
    B = 1000: the last tile is ragged.  N = 0: the one-kernel step; 8: one full work item; 33: a ragged last one;
    200: flag words outside registers, respawns in place.  The whole state is compared after every auto-reset step: a
    lost plane write shows there at once, in the outputs one step later."""
    B, T1, T2, T3 = 1000, 10, 40, 20
    cast = _cast(mode)
    env, ref = _pair(vk, config_class(vk), N, B, mode, seed=1000 + N, auto_reset=False)
    assert np.array_equal(env.reset().cpu().numpy(), cast(ref.reset()))
    rng = np.random.RandomState(N + (mode == "fast"))
    idx = np.arange(B)
    events = np.zeros(6, np.int64)
    for t in range(T1 + T2 + T3):
        auto = t >= T1
        ref.auto_reset = auto
        if t == T1:                                       # what the auto-reset steps below rely on
            ticks = ref.state["tick"]
            assert mixed_groups(ticks, B, 8) >= B // 8 // 2 and mixed_groups(ticks, B, 32) >= B // 32 // 2
            _same_state(env, ref, (vk, N, mode, "before the first auto-reset step"))
        a_host, a_dev = _actions(env, rng, mode == "fast")
        env.step(a_dev, auto_reset=auto)
        ref.step(a_host)
        what = (vk, N, mode, t)
        _same_outputs(env, ref, cast, what)
        events += np.bincount(ref.info, minlength=6)
        if auto:
            _same_state(env, ref, what)
        mask = None
        if not auto:
            mask = ref.done != 0
            if t == T1 // 2:
                mask = mask | (idx % 8 == 0) | (rng.rand(B) < 0.3)
        elif t >= T1 + T2 and t % 5 == 4:
            mask = rng.rand(B) < 0.3
        if mask is not None and mask.any():
            _masked_reset(env, ref, mask, cast, what)
    _same_state(env, ref, (vk, N, mode, "final state"))
    env.close()
    assert events[GOAL] + events[WALL] > 0, events
    if N >= 33:
        assert events[NMAC] > 0 and events[CONFLICT] > 0, events
    elif N > 0:
        assert events[CONFLICT] > 0, events


# ------------------------------------------------------------------------------------------------ tick patterns
def _tick_pattern(name, B, rng):
    i = np.arange(B)
    odd = {"alternating": i % 2 == 1,
           "lane0_odd": i % 8 == 0,                    # lane 0 of every group on the other plane than its 7 neighbours
           "lane7_odd": i % 8 == 7,
           "random": rng.rand(B) < 0.5,
           "tile_uniform": (i // 32) % 2 == 1}[name]   # the control: every tile on one plane
    return (2 * rng.randint(1, 1 << 20, B) + odd).astype(np.uint32)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("pattern", ["alternating", "lane0_odd", "lane7_odd", "random", "tile_uniform"])
@pytest.mark.parametrize("vk", ["env2", "her"])
def test_tick_patterns_auto_reset_vs_oracle(vk, pattern, mode):
    """Ticks set with set_state after reset, then 10 auto-reset steps; state and outputs after every step."""
    B, N = 1000, 80
    cast = _cast(mode)
    env, ref = _pair(vk, config_class(vk), N, B, mode, seed=7, auto_reset=True)
    assert np.array_equal(env.reset().cpu().numpy(), cast(ref.reset()))
    ticks = _tick_pattern(pattern, B, np.random.RandomState(len(pattern)))
    if pattern == "tile_uniform":
        assert mixed_groups(ticks, B, 32) == 0 and len(set((ticks[::32] & 1).tolist())) == 2
    else:
        assert mixed_groups(ticks, B, 8) >= B // 8 // 2
    _set_both(env, ref, {"tick": ticks})
    _same_state(env, ref, (vk, pattern, mode, "after set_state"))
    assert np.array_equal(env.observe().cpu().numpy(), cast(ref.observe()))
    rng = np.random.RandomState(3)
    for t in range(10):
        a_host, a_dev = _actions(env, rng, mode == "fast")
        env.step(a_dev)
        ref.step(a_host)
        what = (vk, pattern, mode, t)
        _same_outputs(env, ref, cast, what)
        _same_state(env, ref, what)
    env.close()


# ------------------------------------------------------------------------------------------------ ticks past 2^31
# within a tile the envs share a parity (the discard above is not what this exercises) but not a sign bit
HIGH_EVEN = np.array([2**31 - 2, 2**31, 2**32 - 2, 0], np.uint32)
HIGH_ODD = np.array([2**31 - 1, 2**31 + 1, 2**32 - 1, 1], np.uint32)


@pytest.mark.parametrize("auto", [True, False])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("per_env", [2, 6])
@pytest.mark.parametrize("vk,N", [(vk, n) for vk in ("env2", "d9her", "mctsrnd") for n in (80, 200)])
def test_ticks_past_2p31_respawns_vs_oracle(vk, N, per_env, mode, auto):
    """Ticks from {2^31 - 2 .. 2^31 + 1, 2^32 - 2, 2^32 - 1, 0, 1}: the queued respawns and the auto-reset spawns of
    such an env use its tick, and the tick wraps at 2^32.  `per_env` intruders of every env sit at x = W - 0.25 moving
    +1 px per step, so they leave the map in the first step: 2 per env fit a tile's respawn list (128 records), 6 per env
    overflow it and the rest respawn in place (N = 200: all in place).  Every fifth ownship sits on its goal."""
    B = 600
    cast = _cast(mode)
    env, ref = _pair(vk, config_class(vk), N, B, mode, seed=31 + N, auto_reset=auto)
    env.reset()
    ref.reset()
    st = {k: v.copy() for k, v in ref.state.items()}
    b = np.arange(B)
    st["tick"] = np.where((b // 32) % 2 == 0, HIGH_EVEN[b % 4], HIGH_ODD[b % 4]).astype(np.uint32)
    assert mixed_groups(st["tick"], B, 32) == 0 and (st["tick"] >= 2**31).sum() >= B // 2
    W = float(ref.cfg.window_width)
    rng = np.random.RandomState(per_env + N)
    planted = np.stack([rng.choice(N, per_env, replace=False) for _ in range(B)])
    own_y = st["own_pos"][:, 1].astype(np.float64)
    y = np.where(own_y < 400, own_y + 300, own_y - 300).astype(np.float32).astype(np.float64)   # 300 px away: no conflict
    for k in range(per_env):
        i = planted[:, k]
        st["ipos"][b, i] = np.stack([np.full(B, W - 0.25), y], -1)
        st["ivel"][b, i] = (1.0, 0.0)
        st["ipos_is_f64"][b, i] = 0
        st["iflag"][b, i] = 0
        if ref.cfg.intruder_turns:
            st["ihs"][b, i] = (0.0, 1.0)                   # heading 0, speed 1: the velocity above
    goal_envs = b % 5 == 0
    st["goal"][goal_envs] = st["own_pos"][goal_envs]
    _set_both(env, ref, st)
    _same_state(env, ref, (vk, N, mode, "after set_state"))
    assert np.array_equal(env.observe().cpu().numpy(), cast(ref.observe()))
    arng = np.random.RandomState(5)
    for t in range(6):
        a_host, a_dev = _actions(env, arng, mode == "fast")
        env.step(a_dev, auto_reset=auto)
        ref.step(a_host)
        what = (vk, N, per_env, mode, auto, t)
        _same_outputs(env, ref, cast, what)
        _same_state(env, ref, what)
        if t == 0:
            px = ref.state["ipos"][b[:, None], planted, 0]
            assert np.all(px <= W), what                   # every planted intruder left the map and was replaced
            assert np.count_nonzero(ref.info[goal_envs] == GOAL) >= goal_envs.sum() // 2, what
        if not auto and ref.done.any():
            _masked_reset(env, ref, ref.done != 0, cast, what)
    wrapped = np.isin(st["tick"], [2**32 - 2, 2**32 - 1])
    assert np.all(ref.state["tick"][wrapped] < 100)       # (wrapped; the device ticks are compared above)
    env.close()


# ------------------------------------------------------------------------------------------------ the bench shape
def test_bench_shape_half_masked_reset_then_auto_reset_vs_oracle():
    """65,536 envs x 80 intruders, env2, FAST: a masked reset of a random half, then 3 auto-reset steps.  The 42 MB
    position plane does not stay in the L2 between steps at this size."""
    vk, N, B = "env2", 80, 65536
    cast = _cast("fast")
    env, ref = _pair(vk, config_class(vk), N, B, "fast", seed=99, auto_reset=True)
    assert np.array_equal(env.reset().cpu().numpy(), cast(ref.reset()))
    rng = np.random.RandomState(12)
    _masked_reset(env, ref, rng.rand(B) < 0.5, cast, "masked reset")
    assert mixed_groups(ref.state["tick"], B, 8) >= B // 8 // 2
    for t in range(3):
        a_host, a_dev = _actions(env, rng, True)
        env.step(a_dev)
        ref.step(a_host)
        _same_outputs(env, ref, cast, t)
        _same_state(env, ref, t)
    env.close()


# ------------------------------------------------------------------------------------------------ tape handles
@pytest.mark.parametrize("vk", sorted(vk for vk, n in GOLDEN_CASES if n == 80))
def test_golden_replay_fast_auto_reset_vs_oracle(vk):
    """The fast golden replay at N = 80 with auto-reset on odd steps and masked resets after even ones, from start
    ticks on both planes within each 8-env group (a tape handle draws from its tape: the tick only picks the plane).
    Flags and draw counts equal the reference's, every bit the oracle twin's."""
    from oracle import oracle as orc
    g = load_trace(vk, 80)
    B = g["tape"].shape[0]
    tape = np.nan_to_num(g["tape"], nan=0.0)
    env = make_gpu(vk, 80, B, "fast", "tape")
    ref = make_oracle(vk, 80, B, 0, orc.TRIG_SHARED, tape=tape, f32=True)
    cast = _cast("fast")
    st = golden_state(g, "s0_")
    st["ipos"] = st["ipos"].astype(np.float32).astype(np.float64)
    st["ipos_is_f64"][...] = 0
    st["tick"] = (np.arange(B) % 3 == 0).astype(np.uint32)
    assert mixed_groups(st["tick"], B, 8) > 0
    _set_both(env, ref, st)
    env.set_tape(tape, cursor=np.broadcast_to(g["cur_reset0"], (B,)))
    ref.cursor[...] = g["cur_reset0"]
    acts = golden_actions(vk, g)
    if env.continuous:
        acts = acts.astype(np.float32).astype(np.float64)
    resets = 0
    for t in range(acts.shape[1]):
        auto = t % 2 == 1
        ref.auto_reset = auto
        what = "%s step %d" % (vk, t)
        env.step(gpu_actions(env, acts[:, t]), auto_reset=auto)
        ref.step(acts[:, t])
        assert np.array_equal(env.info.cpu().numpy(), g["event"][:, t]) and np.array_equal(env.done.cpu().numpy(), g["done"][:, t]), what
        _same_outputs(env, ref, cast, what)
        _same_state(env, ref, what)
        resets += int(ref.done.sum())
        if not auto:
            assert np.array_equal(env.tape_cursor.cpu().numpy(), g["cur_after"][:, t]), what
            if ref.done.any():
                _masked_reset(env, ref, ref.done != 0, cast, what)
        assert np.array_equal(env.tape_cursor.cpu().numpy(), g["cur_after_reset"][:, t]), what
        assert np.array_equal(env.tape_cursor.cpu().numpy(), ref.cursor), what
    assert resets > 0
    env.close()
