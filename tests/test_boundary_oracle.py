"""States whose decisive quantity sits exactly on a chosen side of a threshold, and the oracle checked at them.

The kernels do not always perform the reference's operation.  They compare squared distances with a pre-squared
threshold (sq_threshold of csrc/gca_launch.h: the smallest s with sqrt(s) >= thr) instead of `sqrt(s) < thr`, test the
map on f32 bit patterns instead of `0 <= x <= W`, and so on.  Each shortcut agrees with the reference everywhere, by an
argument; where the argument breaks, the two disagree only within about one ulp of the boundary, which seeded rollouts
almost never reach.  This module builds states that land there: a squared distance of X - 2 ... X + 2 ulp (X =
sq_threshold, the f32 or f64 squared distance computed the reference's way), plus thr^2 where it differs from X;
map coordinates 0, W, nextafter(W, +inf), the smallest negative subnormal and +0.0 reached as x + (-x); spawn draws on
either side of initial_min_dist.  The states are the fixtures of tests/test_gpu_boundaries.py.

The tests here pin the oracle itself at those edges against a plain restatement of the reference's lines (NumPy
scalars, exact Fraction arithmetic for the f64 fma), so that the device tests compare against a reference known to
be right there.  test_cases_separate_the_naive_shortcut shows that the case set would catch `s < thr * thr`.
"""
import math
from fractions import Fraction

import numpy as np
import pytest

from helpers import GOLDEN_VARIANTS, config_class
from gca_b200 import abi, variants

F32, F64 = np.float32, np.float64
OWN0 = (400.25, 399.75)            # ownship start: coordinates with spare low bits, so that dx, dy below are not round
GOAL = (700.0, 120.0)              # far from every boundary intruder


# ------------------------------------------------------------------------------- the reference's arithmetic
def sq_threshold(thr, dt):
    """csrc/gca_launch.h sq_threshold restated: smallest s (of dtype dt) with sqrt(s) >= dt(thr)."""
    t = dt(thr)
    if not t > 0:
        return dt(0)
    c = dt(t * t)
    while c > 0 and dt(np.sqrt(c)) >= t:
        c = np.nextafter(c, dt(0))
    while dt(np.sqrt(c)) < t:
        c = np.nextafter(c, dt(np.inf))
    return c


def fma64(a, b, c):
    """fma(a, b, c) in f64: the exact value, rounded once (Fraction -> float rounds to nearest even)."""
    return float(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def s_f32(ox, oy, x, y):
    """Squared f32 distance of np.linalg.norm(own - intruder), f32 operands: fl(fl(dx^2) + fl(dy^2))."""
    dx, dy = F32(ox) - F32(x), F32(oy) - F32(y)
    return F32(dx * dx) + F32(dy * dy)


def s_f64(ox, oy, x, y):
    """Squared f64 distance with an f64 operand: fma(dy, dy, fl(dx^2)) (OpenBLAS ddot tail), exactly rounded."""
    dx, dy = float(ox) - float(x), float(oy) - float(y)
    return fma64(dy, dy, dx * dx)


def lt_ref(s, thr, dt):
    """The reference's `dist < thr`: dist = sqrt(s) in dtype dt, compared with thr taken in dt (NumPy 2 weak scalars)."""
    if dt is F32:
        return bool(F32(np.sqrt(F32(s))) < F32(thr))
    return bool(math.sqrt(float(s)) < float(thr))


def lt_naive(s, thr, dt):
    """The shortcut the kernels must NOT take: s < thr * thr."""
    t = dt(thr)
    return bool(dt(s) < dt(t * t))


def in_map_ref(x, y, W, H):
    """position_range.contains: 0 <= p <= high, Box of f32 bounds."""
    return bool(0.0 <= x <= float(F32(W))) and bool(0.0 <= y <= float(F32(H)))


def ulps(x, k):
    dt = type(x)
    for _ in range(abs(k)):
        x = np.nextafter(x, dt(np.inf) if k > 0 else dt(-np.inf))
    return x


def threshold_targets(thr, dt):
    """X - 2 ... X + 2 ulp around X = sq_threshold(thr), and thr^2 (in dt) where it differs from X."""
    X = sq_threshold(thr, dt)
    t = dt(thr)
    out = [ulps(X, k) for k in range(-2, 3)]
    if dt(t * t) not in out:
        out.append(dt(t * t))
    return out


def place(ox, oy, target, dt, rng, tries=200, fused=True, angles=(0.0, 2 * np.pi)):
    """An intruder position (x, y) of dtype dt whose squared distance from (ox, oy), computed the reference's way for
    that dtype, is exactly `target`: neighbouring representable coordinates around points at distance sqrt(target) in
    the given direction range.  fused=False: the f64 sum of squares without fma (the MCTS model's metric)."""
    r = math.sqrt(float(target))
    k = np.arange(-6, 7)
    for _ in range(tries):
        th = rng.uniform(angles[0], angles[1], 256)
        x0 = (ox + r * np.cos(th)).astype(dt)
        y0 = (oy + r * np.sin(th)).astype(dt)
        xs = (x0[:, None, None] + k[None, :, None] * np.spacing(x0)[:, None, None]).astype(dt)
        ys = (y0[:, None, None] + k[None, None, :] * np.spacing(y0)[:, None, None]).astype(dt)
        xs, ys = np.broadcast_arrays(xs, ys)
        dx, dy = dt(ox) - xs, dt(oy) - ys
        s = dx * dx + dy * dy                      # f32: every operation rounds once, as the reference's
        if dt is F32 or not fused:
            hit = np.argwhere(s == target)
            if len(hit):
                j = tuple(hit[0])
                return dt(xs[j]), dt(ys[j])
        else:                                      # f64: numpy has no fma; screen, then evaluate exactly
            near = np.argwhere(np.abs(s - target) <= 4 * np.spacing(target))
            for j in map(tuple, near):
                if s_f64(ox, oy, xs[j], ys[j]) == target:
                    return F64(xs[j]), F64(ys[j])
    raise AssertionError("no position found for squared distance %r" % target)


# ------------------------------------------------------------------------------- step states
def boundary_config(vk, **over):
    """(Config class, gca_config) of variant vk with the given Config attributes overridden."""
    base = config_class(vk)
    cls = type("Boundary%s" % vk, (base,), over) if over else base
    return cls, variants.make_config(GOLDEN_VARIANTS[vk], cls)


def step_actions(cfg, B):
    """A straight action for every env (the ownship path does not matter, only that it is known)."""
    a = np.zeros((B, 2))
    if cfg.action_kind == abi.ACT_DISCRETE9:
        a[:, 0] = 4
    elif cfg.action_kind in (abi.ACT_DISCRETE3, abi.ACT_DISCRETE3_HEADING):
        a[:, 0] = 1
    return a


def _far_intruders(st, rng, N):
    """Every intruder 130-300 px from the ownship start, inside the map, on dyadic velocities (pos + vel is exact)."""
    B = st["own_pos"].shape[0]
    ang = rng.uniform(0, 2 * np.pi, (B, N))
    rad = rng.uniform(130, 300, (B, N))
    st["ipos"][..., 0] = np.round(OWN0[0] + rad * np.cos(ang))
    st["ipos"][..., 1] = np.round(OWN0[1] + rad * np.sin(ang))
    st["ivel"][...] = rng.randint(-8, 9, (B, N, 2)) / 8.0


def _start_state(B, N, rng):
    from oracle import oracle as orc
    st = orc.empty_state(B, N)
    st["own_pos"][:] = OWN0
    h = rng.uniform(0, 2 * np.pi, B)
    st["own_hs"][:, 0], st["own_hs"][:, 1] = h, 2.0
    st["own_vel"][:, 0] = (2.0 * np.cos(h)).astype(F32)
    st["own_vel"][:, 1] = (2.0 * np.sin(h)).astype(F32)
    st["own_vel_is_f32"][:] = 1
    st["goal"][:] = GOAL
    _far_intruders(st, rng, N)
    return st


def own_after_step(cfg, st, actions, seed, fast):
    """The ownship's f32 position after one oracle step from st (it does not depend on the intruders)."""
    from oracle import oracle as orc
    B, N = st["ipos"].shape[:2]
    ref = orc.OracleEnv(cfg, B, N, draws=1, trig=orc.TRIG_SHARED, seed=seed, f32_positions=fast)
    for k, v in st.items():
        ref.state[k][...] = v
    ref.step(actions)
    return ref.state["own_pos"].copy()


def threshold_plan(cfg, N, dt):
    """Per-env list of (intruder index, target squared distance) pairs.  One boundary intruder per env for every
    (threshold, target) at rotating indices, plus envs where two intruders straddle the NMAC boundary in either
    order (`nmac &= conf` and the stop at the first NMAC, Q9)."""
    sep, nmac = cfg.minimum_separation, cfg.nmac_dist
    plan = []
    for rep in range(2):
        for thr in (sep, nmac):
            for t in threshold_targets(thr, dt):
                plan.append([((len(plan) * 5 + rep) % N, t)])
    Xn = sq_threshold(nmac, dt)
    Xs = sq_threshold(sep, dt)
    for j in range(4):
        a, b = (j * 3) % N, (j * 3 + 5 + j) % N
        if a == b:
            b = (b + 1) % N
        lo, hi = min(a, b), max(a, b)
        plan.append([(lo, Xn), (hi, ulps(Xn, -1))])          # first in conflict only, the later one is the NMAC
        plan.append([(lo, ulps(Xn, -1)), (hi, ulps(Xn, -2))])  # first NMAC ends the loop: the later one untouched
        plan.append([(lo, ulps(Xs, -1)), (hi, Xn)])          # two conflicts, no NMAC
        plan.append([(lo, Xs), (hi, ulps(Xn, -1))])          # the nearer miss outside, the later one an NMAC
    return plan


def threshold_states(vk, N, mode, seed, sep=None, nmac=None):
    """(cfg class, gca_config, start state, actions, plan, dtype) of the threshold cases for variant vk.
    mode: "fast", "f32" (faithful, f32 intruders) or "f64" (faithful, ipos_is_f64 = 1 for the boundary intruders)."""
    cls, cfg = boundary_config(vk, **({} if sep is None else {"minimum_separation": sep, "NMAC_dist": nmac}))
    dt = F64 if mode == "f64" else F32
    plan = threshold_plan(cfg, N, dt)
    B = len(plan)
    rng = np.random.RandomState(seed)
    st = _start_state(B, N, rng)
    if mode != "fast":                             # some far intruders f64 too: the per-intruder flag words are mixed
        st["ipos_is_f64"][...] = rng.rand(B, N) < 0.3
    acts = step_actions(cfg, B)
    own = own_after_step(cfg, st, acts, seed, mode == "fast")
    for b, items in enumerate(plan):
        for i, target in items:
            x, y = place(own[b, 0], own[b, 1], target, dt, rng)
            st["ipos"][b, i] = (x, y)
            st["ivel"][b, i] = 0.0
            st["ipos_is_f64"][b, i] = dt is F64
            st["iflag"][b, i] = rng.rand() < 0.25       # an intruder already in conflict is not counted again
    return cls, cfg, st, acts, plan, dt, own


def restate_step(cfg, st, own):
    """terminal_reward() of the reference for a state whose intruders do not move and stay in the map (every
    intruder here has zero or dyadic velocity, far from the edges): (info, done, reward, no_conflict, iflag)."""
    B, N = st["ipos"].shape[:2]
    info = np.zeros(B, np.uint8)
    done = np.zeros(B, np.uint8)
    reward = np.zeros(B)
    nc = st["no_conflict"].copy()
    iflag = st["iflag"].copy()
    for b in range(B):
        ox, oy = own[b]
        conflict, ended = False, False
        for i in range(N):
            x = st["ipos"][b, i, 0] + float(st["ivel"][b, i, 0])
            y = st["ipos"][b, i, 1] + float(st["ivel"][b, i, 1])
            if st["ipos_is_f64"][b, i]:
                s, dt = s_f64(ox, oy, x, y), F64
            else:
                s, dt = s_f32(ox, oy, F32(st["ipos"][b, i, 0]) + st["ivel"][b, i, 0],
                              F32(st["ipos"][b, i, 1]) + st["ivel"][b, i, 1]), F32
            if lt_ref(s, cfg.minimum_separation, dt):
                conflict = True
                if not iflag[b, i]:
                    nc[b] += 1
                    iflag[b, i] = 1
                if lt_ref(s, cfg.nmac_dist, dt):
                    info[b], done[b], reward[b] = abi.INFO_NMAC, 1, cfg.r_nmac
                    ended = True
                    break
        if ended:
            continue
        if conflict:
            info[b], reward[b] = abi.INFO_CONFLICT, cfg.r_conflict
            continue
        dg = math.sqrt(s_f64(ox, oy, cfg_goal(st, b)[0], cfg_goal(st, b)[1]))
        assert not dg < cfg.goal_radius
        reward[b] = -dg / 1200 if cfg.shaped_default else cfg.r_default
    return info, done, reward, nc, iflag


def cfg_goal(st, b):
    return st["goal"][b]


def oracle_step(cfg, st, acts, seed, fast, tape=None):
    from oracle import oracle as orc
    B, N = st["ipos"].shape[:2]
    ref = orc.OracleEnv(cfg, B, N, draws=0 if tape is not None else 1, trig=orc.TRIG_SHARED, seed=seed,
                        f32_positions=fast, tape=tape)
    for k, v in st.items():
        ref.state[k][...] = v
    ref.step(acts)
    return ref


# ------------------------------------------------------------------------------- map edges
W_DEFAULT = 800.0


def edge_values(W):
    """Coordinates at and beyond the edges of [0, W] (f32): (value before the step, velocity) pairs whose f32 sum is
    the edge coordinate.  +0.0 is reached as x + v with v = -x."""
    w = F32(W)
    return [(F32(0.0), F32(0.0)), (w, F32(0.0)), (np.nextafter(w, F32(np.inf)), F32(0.0)),
            (F32(-1.4e-45), F32(0.0)), (F32(5.0), F32(-5.0)), (F32(0.75), F32(-0.75)),
            (np.nextafter(F32(0.0), F32(1)), F32(0.0)), (np.nextafter(w, F32(0)), F32(0.0)),
            (w - F32(0.5), F32(0.5)), (w - F32(0.5), np.nextafter(F32(0.5), F32(1)))]


def map_states(vk, N, mode, seed, drift=None):
    """Envs whose intruders land on the map's edges after one step (x, y or both), the rest far inside."""
    cls, cfg = boundary_config(vk, **({} if drift is None else {"position_sigma": drift}))
    assert cfg.position_drift == (drift or 0.0)
    rng = np.random.RandomState(seed)
    ev = edge_values(cfg.window_width)
    evh = edge_values(cfg.window_height)
    combos = [(j, None) for j in range(len(ev))] + [(None, j) for j in range(len(evh))] + \
             [(j, j) for j in range(len(ev))]
    B = 2 * len(combos)
    st = _start_state(B, N, rng)
    d = F32(drift or 0.0)
    for b in range(B):
        jx, jy = combos[b % len(combos)]
        for rep in range(3):                               # three intruders per env, at rotating indices
            i = (b + 5 * rep) % N
            x, vx = ev[jx] if jx is not None else (F32(100.0 + 10 * rep), F32(0.0))
            y, vy = evh[jy] if jy is not None else (F32(700.0 - 10 * rep), F32(0.0))
            # with a drift the velocity is (v + drift) first: pick v so that v + drift is the wanted f32 step
            st["ipos"][b, i] = (x, y)
            st["ivel"][b, i] = (vx - d, vy - d) if d else (vx, vy)
    if drift is not None:                              # v - d + d must give back v exactly
        assert np.array_equal((st["ivel"] + d).astype(F32), st["ivel"] + d)
    return cls, cfg, st, step_actions(cfg, B)


def map_outcome(cfg, st):
    """(f32 positions after `position += velocity (+ drift)`, whether each stays in the map) - the reference's way."""
    d = F32(cfg.position_drift)
    moved = (st["ipos"].astype(F32) + (st["ivel"] + d if cfg.position_drift else st["ivel"])).astype(F32)
    W, H = cfg.window_width, cfg.window_height
    return moved, np.vectorize(lambda x, y: in_map_ref(x, y, W, H))(moved[..., 0], moved[..., 1])


# ------------------------------------------------------------------------------- MCTS roots
def mcts_cfg(**over):
    from Algorithms.MCTS.config_single import Config
    c = abi.make_mcts_config(Config)
    for k, v in over.items():
        setattr(c, k, v)
    return c


def _sincos(h):
    import ctypes as C
    from oracle import oracle as orc
    s, c = C.c_double(), C.c_double()
    orc.lib().gca_oracle_sincos(h, orc.TRIG_SHARED, C.byref(s), C.byref(c))
    return s.value, c.value


def own_path(cfg, ox, oy, vy, heading, frames):
    """Ownship positions of a straight move (action 4) of the noise-free model: speed = clamp(previous vy) (Q23)."""
    s, c = _sincos(heading)
    out = []
    for _ in range(frames):
        sp = max(cfg.min_speed, min(cfg.max_speed, vy))
        vx, vy = sp * c, sp * s
        ox, oy = ox + vx, oy + vy
        out.append((ox, oy))
    return out


def _collinear_inside(fx, fy, X, vy_i, frames):
    """A start (fx, y) straight ahead whose position after `frames` advances by (0, vy_i) is at the largest squared
    distance below X from (fx, fy) that dx = 0 allows: the conflict nearest the separation radius on the line of flight."""
    g = float(np.spacing(fy + 20.0))
    k = int(math.ceil(math.sqrt(X) / g)) + 4
    while True:
        y = fy + k * g - vy_i * frames
        yy = y
        for _ in range(frames):
            yy = yy + vy_i
        dy = yy - fy
        if dy * dy < X:
            return fx, y
        k -= 1


def mcts_boundary_roots(F, n=4, seed=0):
    """Roots of the noise-free model (heading_sigma = speed_sigma = position_sigma = 0) whose straight first move ends,
    at its last sub-frame F - 1, with an intruder (stationary or head-on) or the goal ahead at squared distance
    sep2 - 1, sep2, sep2 + 1 ulp (sep2 = sq_threshold(minimum_separation); the model's metric has no fma).  The ownship
    flies north at max_speed from a start picked so that the rounding of its position sums carries it a little further
    than F * max_speed; "reach" roots put an intruder on that line just inside the separation radius - the case the
    candidate lists' rounding margins exist for.
    Returns (cfg, roots [R, 4 n + 8], per root (kind, ulp offset, whether the margin-free reach drops the intruder))."""
    cfg = mcts_cfg(heading_sigma=0.0, simulate_frame=F)
    v = cfg.max_speed
    X = float(sq_threshold(cfg.minimum_separation, F64))
    reach_bare = cfg.minimum_separation + float(F) * max(abs(cfg.min_speed), abs(cfg.max_speed))
    rng = np.random.RandomState(seed)
    best = None
    for k in range(2000):                          # the start whose F additions of max_speed round up the most
        oy0 = 250.0 + k * 0.0137
        path = own_path(cfg, 400.0, oy0, v, math.pi / 2, F)
        excess = (path[-1][1] - oy0) - F * v
        if best is None or excess > best[0]:
            best = (excess, oy0, path)
    _, oy0, path = best
    fx, fy = path[-1]
    far = [[100.0, 700.0, 0.0, 0.0], [700.0, 700.0, 0.0, 0.0], [100.0, 100.0, 0.0, 0.0], [700.0, 100.0, 0.0, 0.0]]
    roots, info = [], []
    ahead = (math.pi / 2 - 1.0, math.pi / 2 + 1.0)
    cases = [(kind, off) for kind in ("still", "headon", "goal") for off in (-1, 0, 1)] + \
            [("reach", -1), ("reach_headon", -1)]
    for kind, off in cases:
        t = F64(ulps(F64(X), off))
        it = [list(far[i % 4]) for i in range(n)]
        goal = (fx, 60.0)
        drop = None
        if kind == "goal":
            goal = place(fx, fy, t, F64, rng, fused=False, angles=ahead)
        else:
            vi = -1.0 if kind.endswith("headon") else 0.0
            if kind.startswith("reach"):
                x, y = _collinear_inside(fx, fy, X, vi, F)
            else:
                x, y = place(fx, fy - vi * F, t, F64, rng, fused=False, angles=ahead)   # vi * F: exact shift
            yy = float(y)
            for _ in range(F):
                yy = yy + vi
            dx, dy = float(x) - fx, yy - fy
            assert (dx * dx + dy * dy == t) or kind.startswith("reach")
            it[(off + 1) % max(n - 1, 1)] = [float(x), float(y), 0.0, vi]     # never the last intruder (Q22)
            dx0, dy0 = float(x) - 400.0, yy - oy0
            drop = not (dx0 * dx0 + dy0 * dy0 < reach_bare * reach_bare)
        roots.append(sum(it, []) + [400.0, oy0, 0.0, v, v, math.pi / 2, float(goal[0]), float(goal[1])])
        info.append((kind, off, drop))
    return cfg, np.array(roots), info


def rnd_cull_roots(cfg, n, F, margins=(0.0, 0.25, 0.5, 1.0, 2.0, -0.5, -1.0, -2.0, -3.0)):
    """Random-intruder roots: a head-on intruder at root distance own_reach + reach + sep - m for a straight first move
    of F sub-frames, the others far; plus roots outside the cull's stated assumptions (root speed above max_speed, an
    intruder whose speed entry disagrees with |v|)."""
    vmax = max(abs(cfg.max_speed), abs(cfg.min_speed))
    roots = []
    for m in margins:
        for variant in ("plain", "fast_root", "speed_entry"):
            spd = 1.0 if variant == "speed_entry" else 2.0
            D = vmax * F + max(2.0, spd) * F + cfg.minimum_separation - m
            st = np.zeros(6 * n + 8)
            for i in range(n):
                st[6 * i:6 * i + 6] = (60.0 + 7 * i, 740.0 - 3 * i, 0.5, 0.0, 0.5, 0.0)
            j = int(abs(m) * 4) % n
            st[6 * j:6 * j + 6] = (400.0, 100.0 + D, 0.0, -2.0, spd, -math.pi / 2)
            own_speed = 5.0 if variant == "fast_root" else cfg.max_speed
            st[6 * n:] = (400.0, 100.0, 0.0, own_speed, own_speed, math.pi / 2, 400.0, 20.0)
            roots.append(st)
    return np.array(roots)


# ------------------------------------------------------------------------------- tests
def _threshold_sets():
    out = []
    for thr in (555 / 30, 150 / 30, 600 / 30, 3000 / 30, 17.3, 4.3):
        for dt in (F32, F64):
            out.append((thr, dt))
    return out


def test_cases_separate_the_naive_shortcut(capsys):
    """For each threshold and dtype the case set holds squared distances where `s < thr * thr` and `sqrt(s) < thr`
    disagree - wherever they can disagree at all (for 100 both give the same answer: sq_threshold(100) == 100^2)."""
    rng = np.random.RandomState(0)
    report = []
    for thr, dt in _threshold_sets():
        targets = threshold_targets(thr, dt)
        ox, oy = OWN0
        split = 0
        for t in targets:
            x, y = place(ox, oy, t, dt, rng)
            s = s_f32(ox, oy, x, y) if dt is F32 else s_f64(ox, oy, x, y)
            assert s == t
            split += lt_ref(s, thr, dt) != lt_naive(s, thr, dt)
        X = sq_threshold(thr, dt)
        t2 = dt(dt(thr) * dt(thr))
        report.append("thr %-8.5g %s: X %s thr^2 %s, %d of %d cases separate s < thr^2 from sqrt(s) < thr" % (
            thr, dt.__name__, repr(float(X)), repr(float(t2)), split, len(targets)))
        if X != t2:
            assert split >= 1, report[-1]
        else:
            assert split == 0
    for thr in (555 / 30, 150 / 30, 600 / 30, 17.3, 4.3):      # the defaults and the inexact ones: a one-ulp gap
        for dt in (F32, F64):
            assert ulps(sq_threshold(thr, dt), 1) == dt(dt(thr) * dt(thr)), (thr, dt)
    with capsys.disabled():
        print("\n" + "\n".join(report))


@pytest.mark.parametrize("vk", ["env", "her"])
@pytest.mark.parametrize("mode", ["fast", "f32", "f64"])
@pytest.mark.parametrize("N", [16, 13])
@pytest.mark.parametrize("inexact", [False, True], ids=["default", "sep17.3"])
def test_oracle_step_thresholds_equal_restatement(vk, mode, N, inexact):
    sep, nmac = (17.3, 4.3) if inexact else (None, None)
    _, cfg, st, acts, plan, dt, own = threshold_states(vk, N, mode, seed=N + 3 * inexact, sep=sep, nmac=nmac)
    ref = oracle_step(cfg, st, acts, seed=N + 3 * inexact, fast=mode == "fast")
    assert np.array_equal(ref.state["own_pos"], own)
    info, done, reward, nc, iflag = restate_step(cfg, st, own)
    assert np.array_equal(ref.info, info)
    assert np.array_equal(ref.done, done)
    assert np.array_equal(ref.reward, reward)
    assert np.array_equal(ref.state["no_conflict"], nc)
    assert np.array_equal(ref.state["iflag"], iflag)
    # the plan reaches both sides of both thresholds, and the NMAC tie-breaks
    assert set(info.tolist()) == {abi.INFO_NONE, abi.INFO_CONFLICT, abi.INFO_NMAC}
    assert (nc - st["no_conflict"]).max() == 2


@pytest.mark.parametrize("mode", ["fast", "f32"])
@pytest.mark.parametrize("drift", [None, 0.25])
def test_oracle_map_edges_equal_restatement(mode, drift):
    """An intruder that leaves the map is respawned (its position is redrawn); one on the edge stays."""
    vk = "mctsrnd" if drift is not None else "env"
    _, cfg, st, acts = map_states(vk, 16, mode, seed=7, drift=drift)
    ref = oracle_step(cfg, st, acts, seed=7, fast=mode == "fast")
    moved, stays = map_outcome(cfg, st)
    kept = np.all(ref.state["ipos"] == moved, -1)
    assert np.array_equal(kept, stays)
    assert (~stays).sum() > 10 and stays.sum() > 10
    # +0.0 reached as x + (-x), W itself and the smallest positive subnormal are inside
    W = F32(cfg.window_width)
    assert stays[moved[..., 0] == 0].all() and stays[moved[..., 0] == W].all()
    assert not stays[moved[..., 0] == np.nextafter(W, F32(np.inf))].any() and not stays[moved[..., 0] < 0].any()


def spawn_tape(B, first, retry, rest_speed=2.0):
    """Tape rows of gca_reset of the plain env, one intruder: [x, y, speed, heading] of the first draw, then the
    retried positions, then the goal position (reset_env's order)."""
    rows = []
    for b in range(B):
        r = [first[b][0], first[b][1], rest_speed, 1.0]
        for p in retry[b]:
            r += [p[0], p[1]]
        r += [650.0, 650.0]
        rows.append(r)
    L = max(len(r) for r in rows) + 4
    tape = np.zeros((B, L))
    for b, r in enumerate(rows):
        tape[b, :len(r)] = r
    return tape


def spawn_plan(seed, own=(50.0, 50.0)):
    """Reset with the ownship at its fixed reset position (50, 50) and one intruder: the first draw at squared f32
    distance X - 2 ... X + 2 ulp of initial_min_dist = 100 (X == 100^2 here), the retried draw (an f64 position, Q3)
    at f64 squared distance around it; the last retry always far."""
    rng = np.random.RandomState(seed)
    thr = 3000 / 30
    firsts, retries, want = [], [], []
    for t32 in threshold_targets(thr, F32):
        x, y = place(own[0], own[1], t32, F32, rng)
        far = (600.0, 600.0)
        if lt_ref(t32, thr, F32):
            for t64 in threshold_targets(thr, F64):
                rx, ry = place(own[0], own[1], t64, F64, rng)
                firsts.append((float(x), float(y)))
                retries.append([(float(rx), float(ry)), far])
                want.append((t32, t64))
        else:
            firsts.append((float(x), float(y)))
            retries.append([far])
            want.append((t32, None))
    return firsts, retries, want


def test_oracle_spawn_rejection_equals_restatement():
    """reset(): the first draw is kept unless its f32 distance is < initial_min_dist; a retried draw is an f64
    position, rejected while its f64 distance is < initial_min_dist.  Cursor, ipos_is_f64 and the position."""
    from oracle import oracle as orc
    cls, cfg = boundary_config("env")
    firsts, retries, want = spawn_plan(1)
    B = len(firsts)
    tape = spawn_tape(B, firsts, retries)
    ref = orc.OracleEnv(cfg, B, 1, draws=0, trig=orc.TRIG_SHARED, tape=tape)
    ref.reset()
    thr = cfg.initial_min_dist
    seen = set()
    for b in range(B):
        t32, t64 = want[b]
        cur, pos, is64 = 4, firsts[b], 0
        if lt_ref(t32, thr, F32):                       # rejected: the retry, then (if rejected too) the far one
            cur, pos, is64 = 6, retries[b][0], 1
            if lt_ref(t64, thr, F64):
                cur, pos = 8, retries[b][1]
            seen.add(("retry", lt_ref(t64, thr, F64)))
        seen.add(("first", lt_ref(t32, thr, F32)))
        assert ref.cursor[b] == cur + 2, b               # + the goal
        assert ref.state["ipos_is_f64"][b, 0] == is64, b
        want_pos = (float(F32(pos[0])), float(F32(pos[1]))) if not is64 else pos
        assert tuple(ref.state["ipos"][b, 0]) == want_pos, b
    assert seen == {("first", True), ("first", False), ("retry", True), ("retry", False)}


@pytest.mark.parametrize("F", [1, 10, 40])
def test_mcts_boundary_roots_reach_the_edge(F):
    """The oracle's move() sees the conflict / goal exactly for the cases below sep2, and some conflicting intruder
    lies beyond the candidate lists' reach (advance_in_reach) without its rounding margins."""
    from oracle import oracle as orc
    cfg, roots, info = mcts_boundary_roots(F)
    n = (roots.shape[1] - 8) // 4
    drops = 0
    for root, (kind, off, drop) in zip(roots, info):
        _, flags, _, _ = orc.mcts_move(cfg, n, root, 4, trig=orc.TRIG_SHARED)
        want = (abi.MCTS_GOAL if kind == "goal" else abi.MCTS_CONFLICT) if off < 0 else 0
        assert flags == want, (kind, off, flags)
        drops += bool(drop and off < 0)
    assert drops >= (1 if F > 1 else 0), info


@pytest.mark.parametrize("over", [{}, {"min_speed": 3.0, "max_speed": 2.0}, {"min_speed": -1.0}],
                         ids=["default", "min_gt_max", "negative_min"])
@pytest.mark.parametrize("F", [1, 10])
def test_rnd_cull_roots_reach_the_edge(over, F):
    """The head-on random-intruder roots: a straight first move ends inside the separation radius for the intruders
    inside the cull's bound (m > 0) and outside it for those beyond (m < 0), whatever the root's own speed entries."""
    from oracle import oracle as orc
    cfg = mcts_cfg(random_intruders=1, turn_prob=0.0, turn_max_deg=10.0, heading_sigma=0.0, simulate_frame=F, **over)
    margins = (0.0, 0.25, 0.5, 1.0, 2.0, -0.5, -1.0, -2.0, -3.0)
    roots = rnd_cull_roots(cfg, 6, F, margins)
    _, _, fl = orc.mcts_playouts(cfg, 6, roots, 1, 1, first_action=np.full((len(roots), 1), 4, np.int8), seed=4)
    m = np.repeat(margins, 3)
    assert (fl[m > 0, 0] == abi.MCTS_CONFLICT).all() and (fl[m < 0, 0] == 0).all()
