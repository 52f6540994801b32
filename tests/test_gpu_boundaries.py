"""The kernels at the exact values where their shortcut comparisons flip, bit for bit against the oracle.

Fixtures: tests/test_boundary_oracle.py builds the step states (squared distances of X - 2 ... X + 2 ulp around the
pre-squared thresholds, map-edge coordinates, spawn draws on either side of initial_min_dist) and pins the oracle at
them, and builds the MCTS roots.  Every comparison is exact: flags, info, reward, done, observations, the whole
state from get_state and, for tape handles, the draw cursor."""
import math

import numpy as np
import pytest

from helpers import GOLDEN_VARIANTS, assert_state_equal
from test_boundary_oracle import (F32, boundary_config, map_outcome, map_states, mcts_boundary_roots, mcts_cfg,
                                  oracle_step, rnd_cull_roots, spawn_plan, spawn_tape, step_actions, threshold_states)
from gca_b200 import abi

pytestmark = pytest.mark.gpu


def _gpu_env(vk, cls, B, N, mode, draws="philox", seed=0):
    from gca_b200.batched import BatchedAircraftEnv
    return BatchedAircraftEnv(GOLDEN_VARIANTS[vk], B, cls, n_intruders=N, mode=mode, draws=draws, seed=seed)


def _gpu_actions(env, a):
    import torch
    if env.continuous:
        return torch.as_tensor(np.ascontiguousarray(a[:, :2]), device=env.device).to(env.real)
    return torch.as_tensor(np.ascontiguousarray(a[:, 0]).astype(np.int32), device=env.device)


def _compare_step(env, ref, out, fast, what):
    obs, rew, done, info = out
    cast = (lambda x: x.astype(np.float32)) if fast else (lambda x: x)
    D = env.obs_dim
    assert np.array_equal(info.cpu().numpy(), ref.info), what
    assert np.array_equal(done.cpu().numpy(), ref.done), what
    assert np.array_equal(rew.cpu().numpy(), cast(ref.reward)), what
    if D:
        assert np.array_equal(obs.cpu().numpy()[:, :D], cast(ref.obs)), what
    if env.is_goal_env:
        assert np.array_equal(env.achieved.cpu().numpy(), cast(ref.achieved)), what
        assert np.array_equal(env.desired.cpu().numpy(), cast(ref.desired)), what
    assert_state_equal(env.get_state(), ref.state, what, skip=())


def _run_step(vk, cls, cfg, st, acts, mode, seed, tape=None):
    """One step of the device and of the oracle from st; returns (env, ref, step outputs)."""
    fast = mode == "fast"
    B, N = st["ipos"].shape[:2]
    env = _gpu_env(vk, cls, B, N, mode, draws="tape" if tape is not None else "philox", seed=seed)
    env.set_state(st)
    if tape is not None:
        env.set_tape(tape)
    a = acts.astype(np.float32).astype(np.float64) if fast and env.continuous else acts
    out = env.step(_gpu_actions(env, a), auto_reset=False)
    ref = oracle_step(cfg, st, a, seed, fast, tape=tape)
    return env, ref, out


# ------------------------------------------------------------------------------- 1. separation / NMAC
@pytest.mark.parametrize("vk", ["env", "her"])
@pytest.mark.parametrize("mode", ["fast", "f32", "f64"])
@pytest.mark.parametrize("N", [16, 13])
@pytest.mark.parametrize("inexact", [False, True], ids=["default", "sep17.3"])
def test_step_thresholds_bit_exact(vk, mode, N, inexact):
    """Squared distances X - 2 ... X + 2 ulp of the separation and NMAC thresholds (and thr^2), one boundary intruder
    per env at rotating indices, plus pairs straddling the NMAC boundary: fast mode, faithful with f32 intruders,
    faithful with f64 intruders; N = 16 takes the full 8-intruder work items (the OM layouts of env and her), N = 13
    the ragged generic one."""
    sep, nmac = (17.3, 4.3) if inexact else (None, None)
    seed = N + 3 * inexact
    cls, cfg, st, acts, plan, dt, own = threshold_states(vk, N, mode, seed=seed, sep=sep, nmac=nmac)
    env, ref, out = _run_step(vk, cls, cfg, st, acts, "fast" if mode == "fast" else "faithful", seed)
    _compare_step(env, ref, out, mode == "fast", "%s %s N=%d" % (vk, mode, N))
    assert {abi.INFO_NONE, abi.INFO_CONFLICT, abi.INFO_NMAC} <= set(ref.info.tolist())
    env.close()


# ------------------------------------------------------------------------------- 2. map edges
@pytest.mark.parametrize("vk,drift", [("env", None), ("mctsrnd", 0.25)])
@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("N", [16, 13])
def test_intruder_map_edges_bit_exact(vk, drift, mode, N):
    """Intruders landing on 0, W, H, one ulp outside, the smallest negative subnormal, +0.0 reached as x + (-x):
    vectorised (N = 16) and generic (N = 13) paths, and the drift instantiation (position += velocity + sigma)."""
    cls, cfg, st, acts = map_states(vk, N, mode, seed=N, drift=drift)
    env, ref, out = _run_step(vk, cls, cfg, st, acts, mode, seed=N)
    _compare_step(env, ref, out, mode == "fast", "%s %s N=%d" % (vk, mode, N))
    _, stays = map_outcome(cfg, st)
    assert (~stays).sum() > 10 and stays.sum() > 10
    env.close()


def test_set_state_canonicalises_negative_zero_fast():
    """FAST positions are never -0.0 (the map test on f32 bit patterns relies on it): gca_set_state stores +0.0, and
    the step that follows - velocity -0.0, so the sum keeps the sign it was given - equals the oracle's."""
    cls, cfg, st, acts = map_states("env", 16, "fast", seed=3)
    st["ipos"][:, 0] = (-0.0, 300.0)
    st["ipos"][:, 1] = (300.0, -0.0)
    st["ipos"][:, 2] = (-0.0, -0.0)
    st["ivel"][:, :3] = -0.0
    env = _gpu_env("env", cls, st["ipos"].shape[0], 16, "fast", seed=3)
    env.set_state(st)
    got = env.get_state()["ipos"][:, :3]
    assert not np.signbit(got).any() and np.array_equal(got, st["ipos"][:, :3])
    env.close()
    env, ref, out = _run_step("env", cls, cfg, st, acts, "fast", seed=3)
    _compare_step(env, ref, out, True, "negative zero")
    assert not np.signbit(env.get_state()["ipos"][:, :3]).any()
    env.close()


def test_ownship_on_map_edges_bit_exact():
    """The ownship lands exactly on x = 0, W or y = 0, H, or one ulp outside (wall test of env2, settle_own); tape
    draws with zero noise so that the landing point is known."""
    from oracle import oracle as orc
    cls, cfg = boundary_config("env2")
    W, H = F32(cfg.window_width), F32(cfg.window_height)
    pi = math.pi
    spots = [(2.0, 300.0, pi), (798.0, 300.0, 0.0), (float(np.nextafter(F32(798), F32(1e9))), 300.0, 0.0),
             (float(np.nextafter(F32(2), F32(0))), 300.0, pi), (300.0, 2.0, -pi / 2), (300.0, 798.0, pi / 2),
             (300.0, float(np.nextafter(F32(798), F32(1e9))), pi / 2), (300.0, float(np.nextafter(F32(2), F32(0))), -pi / 2),
             (400.0, 400.0, 0.3)]
    N = 16
    B = 4 * len(spots)
    rng = np.random.RandomState(2)
    st = orc.empty_state(B, N)
    for b in range(B):
        x, y, h = spots[b % len(spots)]
        st["own_pos"][b] = (x, y)
        st["own_hs"][b] = (h, 2.0)
        st["own_vel"][b] = (F32(2.0 * math.cos(h)), F32(2.0 * math.sin(h)))
    st["own_vel_is_f32"][:] = 1
    st["goal"][:] = (420.0, 410.0)
    st["ipos"][..., 0] = np.round(rng.uniform(100, 700, (B, N)))
    st["ipos"][..., 1] = np.round(rng.uniform(100, 700, (B, N)))
    keep = np.hypot(st["ipos"][..., 0] - st["own_pos"][:, None, 0], st["ipos"][..., 1] - st["own_pos"][:, None, 1]) < 60
    st["ipos"][keep] = (450.0, 450.0)
    tape = np.zeros((B, 64))                           # ownship noise 0, 0; nothing respawns
    acts = step_actions(cfg, B)
    for mode in ("fast", "faithful"):
        env, ref, out = _run_step("env2", cls, cfg, st, acts, mode, seed=0, tape=tape)
        _compare_step(env, ref, out, mode == "fast", "ownship edges " + mode)
        assert np.array_equal(env.tape_cursor.cpu().numpy(), ref.cursor)
        own = ref.state["own_pos"]
        for v in (0.0, float(W), float(np.nextafter(W, F32(1e9)))):
            assert (own[:, 0] == v).any() and (own[:, 1] == v).any(), v
        assert (ref.info == abi.INFO_WALL).any() and (ref.info != abi.INFO_WALL).any()
        env.close()


# ------------------------------------------------------------------------------- 3. spawn rejection
@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_reset_spawn_rejection_bit_exact(mode):
    """gca_reset of the plain env (ownship reset at (50, 50)): first draws at f32 squared distance X - 2 ... X + 2
    ulp of initial_min_dist, retried draws at f64 squared distance around it (f64 positions in FAITHFUL mode, Q3)."""
    from oracle import oracle as orc
    cls, cfg = boundary_config("env")
    firsts, retries, want = spawn_plan(1)
    B = len(firsts)
    tape = spawn_tape(B, firsts, retries)
    fast = mode == "fast"
    env = _gpu_env("env", cls, B, 1, mode, draws="tape")
    env.set_tape(tape)
    obs = env.reset().cpu().numpy()
    ref = orc.OracleEnv(cfg, B, 1, draws=0, trig=orc.TRIG_SHARED, tape=tape, f32_positions=fast)
    ref.reset()
    cast = (lambda x: x.astype(np.float32)) if fast else (lambda x: x)
    assert np.array_equal(env.tape_cursor.cpu().numpy(), ref.cursor)
    assert np.array_equal(obs[:, :env.obs_dim], cast(ref.obs))
    assert_state_equal(env.get_state(), ref.state, "reset spawn " + mode, skip=("tick",))
    assert len(set(ref.cursor.tolist())) == 3
    if not fast:
        assert ref.state["ipos_is_f64"].any() and not ref.state["ipos_is_f64"].all()
    env.close()


@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_respawn_rejection_in_step_bit_exact(mode):
    """One step in which an intruder leaves the map and respawns, its draws on either side of initial_min_dist from
    the ownship's post-step position (first draw in f32, the retry in f64)."""
    from oracle import oracle as orc
    cls, cfg = boundary_config("env")
    firsts, retries, want = spawn_plan(2, own=(52.0, 50.0))      # where the ownship is when the intruder respawns
    B = len(firsts)
    N = 3
    st = orc.empty_state(B, N)
    st["own_pos"][:] = (50.0, 50.0)
    st["own_hs"][:] = (0.0, 2.0)
    st["own_vel"][:] = (2.0, 0.0)
    st["own_vel_is_f32"][:] = 1
    st["goal"][:] = (700.0, 700.0)
    st["ipos"][:] = [(700.0, 100.0), (799.5, 400.0), (100.0, 700.0)]
    st["ivel"][:] = [(0.0, 0.0), (1.0, 0.0), (0.0, 0.0)]
    acts = step_actions(cfg, B)
    tape = np.zeros((B, 24))                           # ownship noise 0, 0; then the respawn of intruder 1
    for b in range(B):
        r = [0.0, 0.0, firsts[b][0], firsts[b][1], 2.0, 1.0] + sum((list(p) for p in retries[b]), [])
        tape[b, :len(r)] = r
    fast = mode == "fast"
    probe = oracle_step(cfg, st, acts, 0, fast, tape=tape)
    assert np.array_equal(probe.state["own_pos"], np.broadcast_to(F32((52.0, 50.0)), (B, 2)))
    env, ref, out = _run_step("env", cls, cfg, st, acts, mode, seed=0, tape=tape)
    _compare_step(env, ref, out, fast, "respawn " + mode)
    assert np.array_equal(env.tape_cursor.cpu().numpy(), ref.cursor)
    # first draw kept, one retry, two retries (FAST mode stores a retry rounded to f32: its f64 boundary is not reached)
    cursors = set(ref.cursor.tolist())
    assert cursors == ({6, 8} if fast else {6, 8, 10}), cursors
    env.close()


# ------------------------------------------------------------------------------- 4. MCTS
def _mcts_compare_all(cfg, n, roots, playouts=64, sims=40):
    import torch
    from gca_b200 import mcts
    from oracle import oracle as orc
    R = roots.shape[0]
    # move
    states = torch.as_tensor(roots.copy(), device="cuda")
    flags = mcts.move(states, torch.full((R,), 4, dtype=torch.int32, device="cuda"), cfg).cpu().numpy()
    for r in range(R):
        st, fl, _, _ = orc.mcts_move(cfg, n, roots[r], 4, trig=orc.TRIG_SHARED)
        assert flags[r] == fl, r
        assert np.array_equal(states[r].cpu().numpy(), st), r
    # playouts, first action straight (every other playout random)
    fa = np.full((R, playouts), 4, np.int8)
    fa[:, 1::2] = -1
    flags1 = None
    for depth in (1, 2):
        want_r, want_f, want_fl = orc.mcts_playouts(cfg, n, roots, playouts, depth, first_action=fa, seed=3, root_id0=2)
        got_r, got_f, got_fl = mcts.playouts(torch.as_tensor(roots, device="cuda"), playouts, depth=depth, cfg=cfg,
                                             first_action=torch.as_tensor(fa, device="cuda"), seed=3, root_id0=2)
        assert np.array_equal(got_fl.cpu().numpy(), want_fl), depth
        assert np.array_equal(got_f.cpu().numpy(), want_f), depth
        assert np.array_equal(got_r.cpu().numpy(), want_r), depth
        if depth == 1:
            flags1 = want_fl
    return flags1


@pytest.mark.parametrize("F", [1, 10, 40])
def test_mcts_separation_and_goal_boundary_bit_exact(F):
    """move, the packed playout kernel (position_sigma == 0) and the device search at the last sub-frame's sep2 +- 1
    ulp, for an intruder and for the goal."""
    import torch
    from gca_b200 import mcts
    from oracle import oracle as orc
    cfg, roots, info = mcts_boundary_roots(F)
    n = (roots.shape[1] - 8) // 4
    fl = _mcts_compare_all(cfg, n, roots)[:, 0]                 # depth 1, the straight move
    want = [(abi.MCTS_GOAL if kind == "goal" else abi.MCTS_CONFLICT) if off < 0 else 0 for kind, off, _ in info]
    assert np.array_equal(fl, want)
    sims = 30                                            # > 9: every root child is expanded
    for depth in (1, 2):
        want_b, want_n, want_q, want_a = orc.mcts_search_philox(cfg, n, roots, sims, depth, seed=8, root_id0=1)
        act, cn, cq, ca = mcts.search(torch.as_tensor(roots, device="cuda"), sims, depth, cfg=cfg, seed=8, root_id0=1,
                                      return_children=True)
        assert np.array_equal(ca.cpu().numpy(), want_a)
        assert np.array_equal(cn.cpu().numpy(), want_n)
        assert np.array_equal(cq.cpu().numpy(), want_q)
        assert np.array_equal(act.cpu().numpy(), np.stack([want_b // 3, want_b % 3], -1))


@pytest.mark.parametrize("over", [{}, {"min_speed": 3.0, "max_speed": 2.0}, {"min_speed": -1.0}],
                         ids=["default", "min_gt_max", "negative_min"])
@pytest.mark.parametrize("n,playouts", [(6, 64), (6, 300), (90, 32)], ids=["lane", "warp_p300", "warp_n90"])
@pytest.mark.parametrize("F", [1, 10])
def test_random_intruder_cull_margin_bit_exact(over, n, playouts, F):
    """The cull drops an intruder beyond own_reach + reach + sep + 2 of the root; head-on intruders at that bound
    minus 0 ... 2 px (and just beyond) in the lane kernel (<= 80 intruders, <= 256 playouts) and in
    mcts_playout_kernel<0, true>, with roots and configs outside the cull's assumptions.  The oracle culls nothing."""
    cfg = mcts_cfg(random_intruders=1, turn_prob=0.0, turn_max_deg=10.0, heading_sigma=0.0, simulate_frame=F, **over)
    roots = rnd_cull_roots(cfg, n, F)
    import torch
    from gca_b200 import mcts
    from oracle import oracle as orc
    R = roots.shape[0]
    fa = np.full((R, playouts), 4, np.int8)
    fa[:, 1::3] = -1
    straight = []
    for depth in (1, 2):
        want_r, want_f, want_fl = orc.mcts_playouts(cfg, n, roots, playouts, depth, first_action=fa, seed=4, root_id0=7)
        if depth == 1:
            straight = want_fl[:, 0]
        got_r, got_f, got_fl = mcts.playouts(torch.as_tensor(roots, device="cuda"), playouts, depth=depth, cfg=cfg,
                                             first_action=torch.as_tensor(fa, device="cuda"), seed=4, root_id0=7)
        assert np.array_equal(got_fl.cpu().numpy(), want_fl), depth
        assert np.array_equal(got_f.cpu().numpy(), want_f), depth
        assert np.array_equal(got_r.cpu().numpy(), want_r), depth
    # the straight move reaches the separation radius exactly for the roots inside the bound (m > 0)
    assert (straight == abi.MCTS_CONFLICT).sum() >= 12 and (straight == 0).sum() >= 12


# ------------------------------------------------------------------------------- 5. raster
AXES_AND_DIAGONALS = [(1.0, 0.0), (0.0, 1.0), (-1.0, 0.0), (0.0, -1.0), (1.0, 1.0), (-1.0, 1.0), (1.0, -1.0),
                      (-1.0, -1.0), (0.0, 0.0)]


def raster_edge_state(B, N, seed):
    """Sprite centres on integer, quarter and half-integer coordinates.  Samples sit at half-integer coordinates, so a
    half-integer centre with an axis-aligned sprite puts samples exactly on the half-open quad edge lx = +-16, and a
    centre 18.25 px from a 4 x 4 block's centre (a .75 / .25 fraction) puts that block exactly at the pixel cull's reach.
    Headings and velocity directions on the axes and the diagonals (where |cos| + |sin| and so the cull's slack is
    largest), and zero-velocity intruders (the len == 0 branch)."""
    from oracle import oracle as orc
    rng = np.random.RandomState(seed)
    st = orc.empty_state(B, N)
    fracs = np.array([0.0, 0.25, 0.5, 0.75])
    for b in range(B):
        own = np.array([4 * rng.randint(20, 180) + 2 - 18.25 * (b % 2), 4 * rng.randint(20, 180) + 2 + fracs[b % 4]])
        h = (b % 8) * math.pi / 4
        st["own_pos"][b] = own
        st["own_hs"][b] = (h, 2.0)
        st["own_vel"][b] = (F32(2.0 * math.cos(h)), F32(2.0 * math.sin(h)))
        st["goal"][b] = own + (rng.choice([-16.0, 16.0, 18.25, -18.5, 0.5]), rng.choice([-16.0, 16.0, 18.25, 0.0, 7.5]))
        for i in range(N):
            off = np.array([rng.choice([-16.0, 16.0, -18.25, 18.25, 0.0, 32.0, -33.5]),
                            rng.choice([-16.0, 16.0, -18.25, 18.25, 0.5, 20.0, -24.75])])
            st["ipos"][b, i] = own + off + fracs[rng.randint(4)] * (i % 2)
            vx, vy = AXES_AND_DIAGONALS[(b + i) % len(AXES_AND_DIAGONALS)]
            st["ivel"][b, i] = (1.75 * vx, 1.75 * vy)
    st["own_vel_is_f32"][:] = 1
    return st


@pytest.mark.parametrize("mode", ["fast", "faithful"])
@pytest.mark.parametrize("which", ["reference", "lookalike"])
def test_raster_edges_bit_exact(mode, which):
    """ImageBatch frames of the edge states against the CPU restatement (ref.raster), every pixel."""
    import os
    from gca_b200 import sprites, variants
    from gca_b200.stack import ImageBatch
    from gym_guidance_collision_avoidance_single.envs.config import Config
    from oracle import oracle as orc
    if which == "reference":
        sp = sprites.load_sprites(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sprites"))
    else:
        sp = sprites.default_sprites()
    B, N = 48, 12
    st = raster_edge_state(B, N, seed=5)
    env = ImageBatch(B, Config, n_intruders=N, mode=mode, seed=1, sprites=sp)
    env.reset()
    env.batch.set_state(st)
    env._raster(None)
    got = env.frame().cpu().numpy()[..., 0]
    ref = orc.OracleEnv(variants.make_config("SingleAircraftStackEnv", Config), B, N, draws=1, trig=orc.TRIG_SHARED,
                        seed=1, f32_positions=(mode == "fast"))
    for k, v in st.items():
        ref.state[k][...] = v
    want = ref.raster(sp)
    assert np.array_equal(got, want), np.argwhere(got != want)[:4].tolist()
    assert (want != want[0, 0, 0]).sum() > 1000            # the sprites are drawn, not a blank canvas
    env.close()
