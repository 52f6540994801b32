#!/usr/bin/env python
"""Generate the golden vectors under tests/golden/ from the UNMODIFIED reference.

Runs ONLY in the build container (it imports /root/reference, which does not exist on the
GPU box).  The reference has no tests or fixtures of its own (SURVEY.md section 4), so these
traces - recorded from the executable reference - are what pins the oracle.

What is recorded, per trace (one reference env instance driven alone):
  * the ordered tape of every value the reference pulled from the global numpy stream
    (np.random.uniform / normal / randint are wrapped; values are logged AS RETURNED),
  * the full object state after reset (optionally after an engineered override that puts
    the ownship next to an intruder / the goal / a wall so that the rare branches fire),
  * the action sequence and, per step, (obs, reward, done, info, no_conflict, full state),
  * on done, the VecEnv-style reset (baselines dummy_vec_env.py:52-55) and its obs/state.

Usage:  python tests/golden/make_golden.py            (writes tests/golden/*.npz)
"""
import json
import math
import os
import sys
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("GCA_REFERENCE", "/root/reference")

np.float = float  # alias removed in NumPy>=1.24; PKG/SingleAircraft2Env.py:35 uses it
sys.path[:0] = [os.path.join(HERE, "_gymstub"), REF, os.path.join(REF, "Simulators"),
                os.path.join(REF, "Algorithms", "MCTS")]

from gym_guidance_collision_avoidance_single.envs import (  # noqa: E402
    SingleAircraftEnv, SingleAircraft2Env, SingleAircraftHEREnv, SingleAircraftDiscreteHEREnv, SingleAircraftStackEnv)
from gym_guidance_collision_avoidance_single.envs.config import Config as PkgConfig  # noqa: E402
import SingleAircraftMCTSEnv as mcts_env_mod  # noqa: E402  (Simulators/, uses Simulators/config.py)
import SingleAircraftDiscrete9HEREnv as d9her_mod  # noqa: E402  (Simulators/, nearest-n observation)
import SingleAircraftDiscrete3HEREnv as d3her_mod  # noqa: E402  (Simulators/, + nearest-intruder reward term)
import SingleAircraftEnv as simenv_mod  # noqa: E402  (Simulators/ copy: Config-driven rewards)
import SingleAircraftRandomEnv as rndenv_mod  # noqa: E402  (Simulators/, random ownship start)
import SingleAircraftMCTSRandIntruderEnv as mctsrnd_mod  # noqa: E402  (Simulators/, intruders that turn at random)
import config as SimConfigMod  # noqa: E402
import nodes_single  # noqa: E402
import nodes_single_randintru  # noqa: E402  (6-field intruders that turn at random)
import search_single  # noqa: E402
import config_single  # noqa: E402

INFO_CODE = {"": 0, "n": 1, "c": 2, "g": 3, "w": 4, "m": 5}


# ----------------------------------------------------------------------------- tape recorder
class Tape(object):
    """Wraps the global-stream entry points the hot path uses (SURVEY.md Q1)."""

    def __init__(self):
        self.values = []
        self._orig = {}

    def __enter__(self):
        for name in ("uniform", "normal", "randint", "random"):
            self._orig[name] = getattr(np.random, name)
            setattr(np.random, name, self._wrap(self._orig[name]))
        return self

    def __exit__(self, *exc):
        for name, fn in self._orig.items():
            setattr(np.random, name, fn)

    def _wrap(self, fn):
        def wrapped(*a, **k):
            out = fn(*a, **k)
            self.values.extend(np.ravel(np.asarray(out, dtype=np.float64)).tolist())
            return out
        return wrapped

    @property
    def cursor(self):
        return len(self.values)


# ----------------------------------------------------------------------------- state capture
def snapshot(env, n):
    d = env.drone
    st = {
        "own_pos": np.asarray(d.position, dtype=np.float32).copy(),
        "own_pos_dtype_is_f32": np.uint8(d.position.dtype == np.float32),
        "own_vel": np.asarray(d.velocity, dtype=np.float64).copy(),
        "own_vel_is_f32": np.uint8(d.velocity.dtype == np.float32),
        "own_heading": np.float64(d.heading),
        "own_speed": np.float64(d.speed),
        "goal": np.asarray(env.goal.position, dtype=np.float64).copy(),
        "no_conflict": np.int32(env.no_conflict),
        "steps": np.int32(getattr(env, "steps", 0)),
        "ipos": np.zeros((n, 2), np.float64),
        "ipos_is_f64": np.zeros((n,), np.uint8),
        "ivel": np.zeros((n, 2), np.float32),
        "iflag": np.zeros((n,), np.uint8),
        "ihs": np.zeros((n, 2), np.float64),        # Aircraft.heading, Aircraft.speed (SingleAircraftMCTSRandIntruderEnv)
    }
    assert d.position.dtype == np.float32
    for i, it in enumerate(env.intruder_list):
        st["ipos"][i] = np.asarray(it.position, dtype=np.float64)
        st["ipos_is_f64"][i] = it.position.dtype == np.float64
        assert it.velocity.dtype == np.float32
        st["ivel"][i] = it.velocity
        st["iflag"][i] = bool(it.conflict)
        if hasattr(it, "change_heading"):            # only the random-intruder env keeps using them after __init__
            st["ihs"][i] = (it.heading, it.speed)
    return st


def snapshot_keys():
    return ("own_pos", "own_pos_dtype_is_f32", "own_vel", "own_vel_is_f32", "own_heading", "own_speed", "goal",
            "no_conflict", "steps", "ipos", "ipos_is_f64", "ivel", "iflag", "ihs")


def obs_arrays(variant, ob):
    """Flatten an observation into (obs f64[D], achieved f64[2], desired f64[2], achieved_is_f32)."""
    if isinstance(ob, dict):
        ag = ob["achieved_goal"]
        return (np.asarray(ob["observation"], np.float64), np.asarray(ag, np.float64),
                np.asarray(ob["desired_goal"], np.float64), np.uint8(ag.dtype == np.float32))
    return np.asarray(ob, np.float64), np.zeros(2), np.zeros(2), np.uint8(0)


# ----------------------------------------------------------------------------- engineered starts
def override(env, kind, rng, n):
    """Move reference objects (keeping the reference's dtypes) so rare branches fire early."""
    d = env.drone
    if kind == "plain":
        return
    if kind == "mid":                       # mid-map ownship: spawn rejections become likely
        d.position[:] = np.float32(rng.uniform(150, 650, 2))
        d.heading = float(rng.uniform(0, 2 * math.pi))
    elif kind == "near_intruder" and n > 0:  # conflict / NMAC within a few steps
        k = int(rng.randint(n))
        it = env.intruder_list[k]
        r = rng.uniform(0.0, 30.0)
        th = rng.uniform(0, 2 * math.pi)
        d.position[:] = (np.asarray(it.position, np.float64) + r * np.array([math.cos(th), math.sin(th)])).astype(np.float32)
        d.heading = float(rng.uniform(0, 2 * math.pi))
    elif kind == "near_goal":                # goal reached within a few steps
        r = rng.uniform(0.0, 45.0)
        th = rng.uniform(0, 2 * math.pi)
        d.position[:] = np.float32(rng.uniform(100, 700, 2))
        env.goal.position = np.asarray(d.position, np.float64) + r * np.array([math.cos(th), math.sin(th)])
        d.heading = float(th + rng.normal(0, 0.3))
    elif kind == "near_wall":                # ownship leaves the map (wall rule of 2Env / DiscreteHER)
        side = int(rng.randint(4))
        p = rng.uniform(50, 750, 2)
        off = rng.uniform(0.0, 6.0)
        if side == 0:
            p[0], h = off, math.pi
        elif side == 1:
            p[0], h = 800 - off, 0.0
        elif side == 2:
            p[1], h = off, -math.pi / 2
        else:
            p[1], h = 800 - off, math.pi / 2
        d.position[:] = np.float32(p)
        d.heading = float(h + rng.normal(0, 0.2))
    elif kind == "edge_intruders" and n > 0:  # intruders about to leave the map -> respawn path
        d.position[:] = np.float32(rng.uniform(250, 550, 2))
        for it in env.intruder_list[: max(1, n // 2)]:
            vx, vy = float(it.velocity[0]), float(it.velocity[1])
            p = rng.uniform(50, 750, 2)
            if abs(vx) > abs(vy):
                p[0] = 800 - rng.uniform(0, 5) if vx > 0 else rng.uniform(0, 5)
            else:
                p[1] = 800 - rng.uniform(0, 5) if vy > 0 else rng.uniform(0, 5)
            if it.position.dtype == np.float32:
                it.position[:] = np.float32(p)
            else:
                it.position = np.asarray(p, np.float64)
    elif kind == "near_maxsteps":            # StackEnv: `steps >= max_steps` fires inside the trace (:134-136)
        env.steps = int(env.max_steps - rng.randint(2, 30))
        d.position[:] = np.float32(rng.uniform(150, 650, 2))
    # anything else (e.g. near_intruder with n == 0): leave the reset state alone


VARIANTS = {
    # name: (class, config class to set N on, action kind)
    "env": (SingleAircraftEnv, PkgConfig, "d9"),
    "env2": (SingleAircraft2Env, PkgConfig, "c2"),
    "her": (SingleAircraftHEREnv, PkgConfig, "c2"),
    "dher": (SingleAircraftDiscreteHEREnv, PkgConfig, "d3"),
    "mcts": (mcts_env_mod.SingleAircraftEnv, SimConfigMod.Config, "t33"),
    "d9her": (d9her_mod.SingleAircraftDiscrete9HEREnv, SimConfigMod.Config, "d9"),
    "d3her": (d3her_mod.SingleAircraftDiscrete3HEREnv, SimConfigMod.Config, "d3"),
    "simenv": (simenv_mod.SingleAircraftEnv, SimConfigMod.Config, "d9"),
    "rndenv": (rndenv_mod.SingleAircraftRandomEnv, SimConfigMod.Config, "d9"),
    "mctsrnd": (mctsrnd_mod.SingleAircraftEnv, SimConfigMod.Config, "t33"),
    # the dynamics of the image env (max_steps rule, non-terminal wall penalty, goal +10000); its observation is the GL
    # frame, which cannot be drawn here: _get_ob is replaced by an empty array so that render() is never called
    "stack": (SingleAircraftStackEnv, PkgConfig, "d9"),
}
# np.argpartition(dist_array, Config.n) of the nearest-n observation needs more than n = 4 intruders
PLANS = {"stack": {0: (3, 40), 3: (6, 40), 80: (3, 30)}, "mctsrnd": {1: (4, 40), 3: (5, 40), 80: (3, 30)}, "simenv": {3: (3, 40), 80: (2, 25)}, "rndenv": {3: (3, 40), 80: (2, 25)}, "d9her": {5: (5, 40), 12: (5, 40), 80: (3, 30)}, "d3her": {5: (5, 40), 12: (5, 40), 80: (3, 30)}}


def sample_action(kind, rng):
    if kind == "d9":
        return np.array([rng.randint(9), 0], np.float64)
    if kind == "d3":
        return np.array([rng.randint(3), 0], np.float64)
    if kind == "t33":
        return np.array([rng.randint(3), rng.randint(3)], np.float64)
    a = rng.uniform(-1, 1, 2)
    # exercise the exact bounds of Box(-1, 1) now and then
    if rng.uniform() < 0.1:
        a[int(rng.randint(2))] = float(rng.choice([-1.0, 1.0, 0.0]))
    return a.astype(np.float64)


def ref_action(kind, a):
    if kind in ("d9", "d3"):
        return int(a[0])
    if kind == "t33":
        return (int(a[0]), int(a[1]))
    return np.array(a, dtype=np.float64)


def info_code(info):
    if isinstance(info, dict):
        info = info.get("result", "")
    if not isinstance(info, str):            # Discrete3HER returns dist_nearest_intruder in place of info (:178)
        return 255
    return INFO_CODE[info]


def run_trace(variant, n, seed, kind, T):
    cls, cfg, akind = VARIANTS[variant]
    cfg.intruder_size = n
    rng = np.random.RandomState((1000003 * seed + 17) % (2 ** 32))   # private: never touches the global stream
    np.random.seed(seed)
    env = cls()                                          # HER ctors reset() here; draws discarded
    if variant == "stack":
        env._get_ob = lambda: np.zeros(0)                # (the frame: make_stack_frame_golden)
    rec = {k: [] for k in ("actions", "obs", "ag", "dg", "reward", "reward_is_int", "done", "info", "event", "nearest",
                           "reward_is_f32",
                           "no_conflict", "cur_before", "cur_after", "cur_after_reset", "reset_obs",
                           "reset_ag", "reset_dg")}
    states_after, states_reset, reset_steps = [], [], []
    # observe (not alter) the raw event string even where the variant hides it (DiscreteHER returns {})
    inner = env._terminal_reward
    last_event = [""]

    def spy():
        out = inner()
        last_event[0] = out[2]
        return out
    env._terminal_reward = spy
    with Tape() as tape:
        ob0 = env.reset()
        cur_reset0 = tape.cursor
        override(env, kind, rng, n)
        state0 = snapshot(env, n)
        ob0 = env._get_ob()
        o0, ag0, dg0, ag_f32 = obs_arrays(variant, ob0)
        for _ in range(T):
            a = sample_action(akind, rng)
            rec["actions"].append(a)
            rec["cur_before"].append(tape.cursor)
            ob, r, done, info = env.step(ref_action(akind, a))
            rec["cur_after"].append(tape.cursor)
            o, ag, dg, _ = obs_arrays(variant, ob)
            rec["obs"].append(o); rec["ag"].append(ag); rec["dg"].append(dg)
            rec["reward"].append(np.float64(r))
            rec["reward_is_int"].append(np.uint8(isinstance(r, int)))
            rec["done"].append(np.uint8(bool(done)))
            rec["info"].append(np.uint8(info_code(info)))
            rec["nearest"].append(np.float64(info) if not isinstance(info, (str, dict)) else np.float64(np.nan))
            rec["reward_is_f32"].append(np.uint8(isinstance(r, np.float32)))
            rec["event"].append(np.uint8(INFO_CODE[last_event[0]]))
            rec["no_conflict"].append(np.int32(env.no_conflict))
            states_after.append(snapshot(env, n))
            if done:
                rob = env.reset()
                reset_steps.append(len(states_after) - 1)
                states_reset.append(snapshot(env, n))
            ro, rag, rdg, _ = obs_arrays(variant, rob if done else ob)
            rec["reset_obs"].append(ro); rec["reset_ag"].append(rag); rec["reset_dg"].append(rdg)
            rec["cur_after_reset"].append(tape.cursor)
        tape_vals = np.asarray(tape.values, np.float64)
    out = {k: np.asarray(v) for k, v in rec.items()}
    out["tape"] = tape_vals
    out["cur_reset0"] = np.int64(cur_reset0)
    out["obs0"], out["ag0"], out["dg0"], out["ag_is_f32"] = o0, ag0, dg0, ag_f32
    for k in state0:
        out["s0_" + k] = state0[k]
        out["sa_" + k] = np.asarray([s[k] for s in states_after])
    out["_reset_steps"] = reset_steps
    out["_states_reset"] = states_reset
    return out


def stack_traces(traces):
    keys = [k for k in traces[0].keys() if not k.startswith("_")]
    L = max(len(t["tape"]) for t in traces)
    out = {}
    # states after VecEnv-style resets, as a compact list: sr_where[j] = (trace, step)
    where = [(ti, st) for ti, t in enumerate(traces) for st in t["_reset_steps"]]
    flat = [s for t in traces for s in t["_states_reset"]]
    out["sr_where"] = np.asarray(where, np.int32).reshape(-1, 2)
    for k in snapshot_keys():
        out["sr_" + k] = np.asarray([s[k] for s in flat]) if flat else np.zeros((0,))
    for k in keys:
        if k == "tape":
            arr = np.full((len(traces), L), np.nan)
            for i, t in enumerate(traces):
                arr[i, : len(t["tape"])] = t["tape"]
            out[k] = arr
        else:
            out[k] = np.asarray([t[k] for t in traces])
    out["tape_len"] = np.asarray([len(t["tape"]) for t in traces], np.int64)
    return out


# Every golden file stays under 1 MB.  Where the traces of a plan do not fit, only those listed are stored: each
# scenario kind, each event and each VecEnv-style reset of the whole plan is among them.
TRACE_SUBSET = {("mctsrnd", 80): (0, 1, 4, 7, 8, 9, 10, 11, 12, 17)}


def select_traces(out, keep):
    """The arrays of stack_traces() for the traces `keep` only: reset records re-indexed, tape padded to the longest."""
    keep = list(keep)
    index = {t: i for i, t in enumerate(keep)}
    rows = [j for j, t in enumerate(out["sr_where"][:, 0]) if t in index]
    L = int(out["tape_len"][keep].max())
    sel = {}
    for k, v in out.items():
        if k == "sr_where":
            sel[k] = np.asarray([[index[t], s] for t, s in v[rows]], np.int32).reshape(-1, 2)
        elif k.startswith("sr_"):
            sel[k] = v[rows]
        elif k == "tape":
            sel[k] = v[keep, :L]
        else:
            sel[k] = v[keep]
    return sel


def savez_lzma(fn, **arrays):
    """np.savez with LZMA-compressed members (np.load reads them like any .npz; smaller than savez_compressed)."""
    with zipfile.ZipFile(fn, "w", zipfile.ZIP_LZMA) as z:
        for k, v in arrays.items():
            with z.open(k + ".npy", "w") as f:
                np.lib.format.write_array(f, np.asanyarray(v), allow_pickle=False)


def make_env_goldens():
    plan = {  # N: (traces per kind, steps per trace)
        0: (3, 40), 1: (6, 40), 3: (6, 40), 80: (3, 25),
    }
    kinds = ["plain", "mid", "near_intruder", "near_goal", "near_wall", "edge_intruders"]
    meta = {}
    only = os.environ.get("GCA_GOLDEN_ONLY")
    for variant in VARIANTS:
        if only and variant not in only.split(","):
            continue
        for n, (per_kind, T) in PLANS.get(variant, plan).items():
            traces, kind_ids = [], []
            seed = 100 * n + 7
            for ki, kind in enumerate(kinds + (["near_maxsteps"] if variant == "stack" else [])):
                if n == 0 and kind in ("near_intruder", "edge_intruders"):
                    continue
                for _ in range(per_kind):
                    seed += 1
                    traces.append(run_trace(variant, n, seed, kind, T))
                    kind_ids.append(ki)
            out = stack_traces(traces)
            out["kind_id"] = np.asarray(kind_ids, np.int32)
            if (variant, n) in TRACE_SUBSET:
                out = select_traces(out, TRACE_SUBSET[variant, n])
            fn = os.path.join(HERE, "trace_%s_n%d.npz" % (variant, n))
            savez_lzma(fn, **out)
            counts = np.bincount(out["event"].ravel(), minlength=6).tolist()
            respawn = int((out["cur_after"] - out["cur_before"] > 2).sum())
            f64pos = int(out["sa_ipos_is_f64"].sum())
            meta["%s_n%d" % (variant, n)] = {"traces": len(out["kind_id"]), "steps": T, "info_counts": counts,
                                             "steps_with_respawn": respawn, "f64_pos_intruder_steps": f64pos}
            print(fn, meta["%s_n%d" % (variant, n)])
    return meta


# ----------------------------------------------------------------------------- MCTS forward model
def mcts_roots(n, seed, count, kind_cycle):
    """Raw observations of Simulators/SingleAircraftMCTSEnv to be used as MCTS root states."""
    SimConfigMod.Config.intruder_size = n
    rng = np.random.RandomState(seed)
    np.random.seed(seed)
    roots = []
    for c in range(count):
        env = mcts_env_mod.SingleAircraftEnv()
        env.reset()
        kind = kind_cycle[c % len(kind_cycle)]
        override(env, kind, rng, n)
        if kind == "near_intruder":
            # aim the ownship at one of the intruders the model can see (it ignores the last one, Q22)
            it = env.intruder_list[int(rng.randint(n - 1))]
            r, th = rng.uniform(8.0, 45.0), rng.uniform(0, 2 * math.pi)
            env.drone.position[:] = (np.asarray(it.position, np.float64)
                                     - r * np.array([math.cos(th), math.sin(th)])).astype(np.float32)
            env.drone.heading = float(th + rng.normal(0, 0.15))
        for _ in range(int(rng.randint(0, 4)) if kind != "near_intruder" else 1):
            env.step((int(rng.randint(3)), int(rng.randint(3))))
        roots.append(np.asarray(env._get_ob(), np.float64))
    return np.asarray(roots)


def make_mcts_goldens():
    meta = {}
    kinds = ["plain", "mid", "near_intruder", "near_goal", "near_wall"]
    for n, count in ((3, 20), (80, 10)):
        roots = mcts_roots(n, 4242 + n, count, kinds)
        mv = {k: [] for k in ("root", "action", "tape", "out_state", "hit_wall", "conflict", "reach_goal", "reward")}
        ro = {k: [] for k in ("root", "depth", "tape", "reward")}
        for ri, root in enumerate(roots):
            for a0 in range(3):
                for a1 in range(3):
                    np.random.seed(7000 + 9 * ri + 3 * a0 + a1)
                    with Tape() as tape:
                        s2 = nodes_single.SingleAircraftState(state=root.copy()).move((a0, a1))
                    mv["root"].append(ri); mv["action"].append((a0, a1)); mv["tape"].append(np.asarray(tape.values))
                    mv["out_state"].append(np.asarray(s2.state, np.float64))
                    mv["hit_wall"].append(s2.hit_wall); mv["conflict"].append(s2.conflict)
                    mv["reach_goal"].append(s2.reach_goal); mv["reward"].append(np.float64(s2.reward()))
            for depth in (1, 2, 3):
                for rep in range(3):
                    np.random.seed(9000 + 31 * ri + 7 * depth + rep)
                    node = nodes_single.SingleAircraftNode(nodes_single.SingleAircraftState(state=root.copy()))
                    with Tape() as tape:
                        r = node.rollout(depth)
                    ro["root"].append(ri); ro["depth"].append(depth); ro["tape"].append(np.asarray(tape.values))
                    ro["reward"].append(np.float64(r))

        def pad(lst):
            L = max(len(x) for x in lst)
            arr = np.full((len(lst), L), np.nan)
            for i, x in enumerate(lst):
                arr[i, : len(x)] = x
            return arr, np.asarray([len(x) for x in lst], np.int64)
        out = {"roots": roots}
        for name, d in (("mv", mv), ("ro", ro)):
            for k, v in d.items():
                if k == "tape":
                    out[name + "_tape"], out[name + "_tape_len"] = pad(v)
                else:
                    out[name + "_" + k] = np.asarray(v)
        # whole searches (tree policy + expand + rollout + backprop), small budget to keep the tape small
        bs = {k: [] for k in ("root", "sims", "depth", "tape", "action", "child_n", "child_q", "child_action")}
        for ri, root in enumerate(roots[: (6 if n == 3 else 2)]):
            for sims, depth in ((30, 2), (100, 3)) if n == 3 else ((20, 2),):
                np.random.seed(12000 + 13 * ri + sims)
                node = nodes_single.SingleAircraftNode(nodes_single.SingleAircraftState(state=root.copy()))
                with Tape() as tape:
                    best = search_single.MCTS(node).best_action(sims, depth)
                bs["root"].append(ri); bs["sims"].append(sims); bs["depth"].append(depth)
                bs["tape"].append(np.asarray(tape.values)); bs["action"].append(best.state.prev_action)
                cn = np.zeros(9); cq = np.zeros(9); ca = np.full((9, 2), -1)
                for ci, c in enumerate(node.children):
                    cn[ci], cq[ci], ca[ci] = c.n, c.q, c.state.prev_action
                bs["child_n"].append(cn); bs["child_q"].append(cq); bs["child_action"].append(ca)
        for k, v in bs.items():
            if k == "tape":
                out["bs_tape"], out["bs_tape_len"] = pad(v)
            else:
                out["bs_" + k] = np.asarray(v)
        fn = os.path.join(HERE, "mcts_n%d.npz" % n)
        np.savez_compressed(fn, **out)
        meta["mcts_n%d" % n] = {"roots": len(roots), "moves": len(mv["root"]), "rollouts": len(ro["root"]),
                                "searches": len(bs["root"]),
                                "move_flags": [int(np.sum(mv["hit_wall"])), int(np.sum(mv["conflict"])), int(np.sum(mv["reach_goal"]))]}
        print(fn, meta["mcts_n%d" % n])
    return meta


def make_mctsrnd_model_goldens():
    """move() and rollout() of Algorithms/MCTS/nodes_single_randintru.py on raw observations of
    Simulators/SingleAircraftMCTSRandIntruderEnv (6 N + 8 values); draw order per intruder and sub-frame:
    normal, normal, random(), [uniform(-10, 10)]."""
    meta = {}
    kinds = ["plain", "mid", "near_intruder", "near_goal", "near_wall"]
    mod = nodes_single_randintru
    for n, count in ((3, 20), (20, 10)):
        SimConfigMod.Config.intruder_size = n
        rng = np.random.RandomState(777 + n)
        np.random.seed(777 + n)
        roots = []
        for c in range(count):
            env = mctsrnd_mod.SingleAircraftEnv()
            env.reset()
            kind = kinds[c % len(kinds)]
            override(env, kind, rng, n)
            if kind == "near_intruder":
                it = env.intruder_list[int(rng.randint(n))]
                r, th = rng.uniform(8.0, 45.0), rng.uniform(0, 2 * math.pi)
                env.drone.position[:] = (np.asarray(it.position, np.float64)
                                         - r * np.array([math.cos(th), math.sin(th)])).astype(np.float32)
                env.drone.heading = float(th + rng.normal(0, 0.15))
            for _ in range(int(rng.randint(0, 4)) if kind != "near_intruder" else 1):
                env.step((int(rng.randint(3)), int(rng.randint(3))))
            roots.append(np.asarray(env._get_ob(), np.float64))
        roots = np.asarray(roots)
        mv = {k: [] for k in ("root", "action", "tape", "out_state", "hit_wall", "conflict", "reach_goal", "reward")}
        ro = {k: [] for k in ("root", "depth", "tape", "reward")}
        for ri, root in enumerate(roots):
            for a0 in range(3):
                for a1 in range(3):
                    np.random.seed(17000 + 9 * ri + 3 * a0 + a1)
                    with Tape() as tape:
                        s2 = mod.SingleAircraftState(state=root.copy()).move((a0, a1))
                    mv["root"].append(ri); mv["action"].append((a0, a1)); mv["tape"].append(np.asarray(tape.values))
                    mv["out_state"].append(np.asarray(s2.state, np.float64))
                    mv["hit_wall"].append(s2.hit_wall); mv["conflict"].append(s2.conflict)
                    mv["reach_goal"].append(s2.reach_goal); mv["reward"].append(np.float64(s2.reward()))
            for depth in (1, 2, 3):
                for rep in range(3):
                    np.random.seed(19000 + 31 * ri + 7 * depth + rep)
                    node = mod.SingleAircraftNode(mod.SingleAircraftState(state=root.copy()))
                    with Tape() as tape:
                        r = node.rollout(depth)
                    ro["root"].append(ri); ro["depth"].append(depth); ro["tape"].append(np.asarray(tape.values))
                    ro["reward"].append(np.float64(r))

        def pad(lst):
            L = max(len(x) for x in lst)
            arr = np.full((len(lst), L), np.nan)
            for i, x in enumerate(lst):
                arr[i, : len(x)] = x
            return arr, np.asarray([len(x) for x in lst], np.int64)
        out = {"roots": roots}
        for name, d in (("mv", mv), ("ro", ro)):
            for k, v in d.items():
                if k == "tape":
                    out[name + "_tape"], out[name + "_tape_len"] = pad(v)
                else:
                    out[name + "_" + k] = np.asarray(v)
        fn = os.path.join(HERE, "mctsrnd_model_n%d.npz" % n)
        np.savez_compressed(fn, **out)
        turns = int(sum(len(t) for t in mv["tape"]))
        meta["mctsrnd_model_n%d" % n] = {"roots": len(roots), "moves": len(mv["root"]), "rollouts": len(ro["root"]),
                                         "move_draws": turns,
                                         "move_flags": [int(np.sum(mv["hit_wall"])), int(np.sum(mv["conflict"])),
                                                        int(np.sum(mv["reach_goal"]))]}
        print(fn, meta["mctsrnd_model_n%d" % n])
    return meta


# ----------------------------------------------------------------------------- StackEnv picture
def _load_rgba(path):
    from PIL import Image
    return np.asarray(Image.open(path).convert("RGBA"), np.uint8)


def render_independent(own_pos, own_heading, goal, ipos, iheading, sprites_rgba, W=800, H=800):
    """An INDEPENDENT software rendition of PKG/SingleAircraftStackEnv.py:179-214 + gym's rendering.Viewer (white
    clear; each sprite a 32x32 textured quad centred on the entity, rotated by heading - pi/2, goal unrotated;
    GL_LINEAR texture filter; GL_SRC_ALPHA / GL_ONE_MINUS_SRC_ALPHA blending into an 8-bit colour buffer; draw order
    ownship, goal, intruders; returned array flipped so that row 0 is y = H).  float64 numpy + scipy.ndimage
    bilinear sampling: shares no code and no arithmetic with csrc/gca_raster_spec.h.  Returns uint8 [H, W, 3]."""
    from scipy import ndimage
    fb = np.full((H, W, 3), 255.0)                                     # row 0 = top of the picture
    def draw(cx, cy, rot, tex):
        texf = tex[::-1].astype(np.float64)                            # row index = v, 0 at the bottom of the image
        x0, x1 = max(int(math.floor(cx - 24)), 0), min(int(math.ceil(cx + 24)), W - 1)
        y0, y1 = max(int(math.floor(cy - 24)), 0), min(int(math.ceil(cy + 24)), H - 1)
        if x0 > x1 or y0 > y1:
            return
        X, Y = np.meshgrid(np.arange(x0, x1 + 1) + 0.5, np.arange(y0, y1 + 1) + 0.5)   # pixel centres, world units
        dx, dy = X - cx, Y - cy
        c, s_ = math.cos(rot), math.sin(rot)
        lx, ly = c * dx + s_ * dy, -s_ * dx + c * dy                   # quad-local coordinates
        inside = (lx >= -16) & (lx < 16) & (ly >= -16) & (ly < 16)
        coords = np.stack([ly + 15.5, lx + 15.5])                      # texel centres at integer + 0.5
        samp = np.stack([ndimage.map_coordinates(texf[:, :, k], coords, order=1, mode="nearest") for k in range(4)], -1)
        alpha = samp[..., 3:4] / 255.0
        rows = (H - 1) - np.arange(y0, y1 + 1)                         # world row y -> picture row
        dst = fb[rows[:, None], np.arange(x0, x1 + 1)[None, :]]
        out = np.rint(samp[..., :3] * alpha + dst * (1.0 - alpha))     # 8-bit colour buffer after every draw
        fb[rows[:, None], np.arange(x0, x1 + 1)[None, :]] = np.where(inside[..., None], out, dst)
    draw(float(own_pos[0]), float(own_pos[1]), own_heading - math.pi / 2, sprites_rgba[0])
    draw(float(goal[0]), float(goal[1]), 0.0, sprites_rgba[1])
    for p, h in zip(ipos, iheading):
        draw(float(p[0]), float(p[1]), h - math.pi / 2, sprites_rgba[2])
    return np.clip(fb, 0, 255).astype(np.uint8)


def make_stack_frame_golden():
    """Frames of the image env: states taken from the unmodified reference StackEnv (reset + a few steps, engineered
    starts so that sprites overlap each other and the map border), drawn with the reference's own PNG sprites by
    render_independent(), then the reference's preprocess_frame (real cv2: RGB2GRAY + INTER_AREA 4x)."""
    import cv2
    img_dir = os.path.join(REF, "gym_guidance_collision_avoidance_single", "envs", "images")
    sprites = np.stack([_load_rgba(os.path.join(img_dir, f)) for f in ("aircraft.png", "goal.png", "intruder.png")])
    rec = {k: [] for k in ("own_pos", "own_hs", "goal", "ipos", "ivel", "iheading", "n", "frame")}
    NMAX = 80
    rng = np.random.RandomState(31)
    for n, kind, seed, steps in ((0, "plain", 1, 0), (3, "plain", 2, 3), (3, "near_intruder", 3, 2), (3, "near_goal", 4, 1),
                                 (3, "near_wall", 5, 2), (12, "edge_intruders", 6, 4), (80, "plain", 7, 0),
                                 (80, "mid", 8, 5), (80, "near_intruder", 9, 3), (80, "edge_intruders", 10, 6)):
        PkgConfig.intruder_size = n
        np.random.seed(1000 + seed)
        env = SingleAircraftStackEnv()
        env._get_ob = lambda: np.zeros(0)
        env.reset()
        override(env, kind, rng, n)
        for _ in range(steps):
            _, _, done, _ = env.step(int(rng.randint(9)))
            if done:
                env.reset()
        d = env.drone
        ipos = np.zeros((NMAX, 2)); ivel = np.zeros((NMAX, 2), np.float32); ihd = np.zeros(NMAX)
        for i, it in enumerate(env.intruder_list):
            ipos[i], ivel[i], ihd[i] = np.asarray(it.position, np.float64), it.velocity, it.heading
        rgb = render_independent(d.position, d.heading, env.goal.position, ipos[:n], ihd[:n], sprites)
        frame = env.preprocess_frame(rgb)[:, :, 0]                     # PKG/SingleAircraftStackEnv.py:104-108, real cv2
        rec["own_pos"].append(np.asarray(d.position, np.float32)); rec["own_hs"].append((d.heading, d.speed))
        rec["goal"].append(np.asarray(env.goal.position, np.float64)); rec["ipos"].append(ipos); rec["ivel"].append(ivel)
        rec["iheading"].append(ihd); rec["n"].append(n); rec["frame"].append(frame)
    out = {k: np.asarray(v) for k, v in rec.items()}
    np.savez_compressed(os.path.join(HERE, "stack_frames.npz"), **out)
    # the sprites themselves, as test vectors (the product never ships them: gca_b200/sprites.py)
    import shutil
    os.makedirs(os.path.join(HERE, "sprites"), exist_ok=True)
    for f in ("aircraft.png", "goal.png", "intruder.png"):
        shutil.copyfile(os.path.join(img_dir, f), os.path.join(HERE, "sprites", f))
        os.chmod(os.path.join(HERE, "sprites", f), 0o644)
    return {"stack_frames": {"frames": len(rec["n"]), "non_white_pixels": [int((f != 255).sum()) for f in rec["frame"]]}}


def make_her_reward_golden():
    """compute_reward of both GoalEnv variants on random + engineered pairs (SURVEY a11)."""
    rng = np.random.RandomState(5)
    PkgConfig.intruder_size = 0
    np.random.seed(3)
    her, dher = SingleAircraftHEREnv(), SingleAircraftDiscreteHEREnv()
    ag_n = rng.uniform(0, 1, (256, 2)); g_n = rng.uniform(0, 1, (256, 2))
    ag_p = rng.uniform(0, 800, (256, 2)); g_p = ag_p + rng.uniform(-30, 30, (256, 2))
    g_p[:8] = ag_p[:8] + np.array([[20.0, 0.0]])          # exactly on the radius
    out = {"ag_n": ag_n, "g_n": g_n, "r_her": her.compute_reward(ag_n, g_n, None),
           "ag_p": ag_p, "g_p": g_p, "r_dher": dher.compute_reward(ag_p, g_p, None),
           "r_her_pix": her.compute_reward(ag_p, g_p, None)}
    np.savez_compressed(os.path.join(HERE, "her_reward.npz"), **out)
    return {"her_reward": {"pairs": 256}}


def make_d9her_reward_golden():
    """compute_reward / compute_input_reward of Simulators/SingleAircraftDiscrete9HEREnv.py:229-277 (scalar calls)."""
    rng = np.random.RandomState(9)
    SimConfigMod.Config.intruder_size = 8
    np.random.seed(4)
    env = d9her_mod.SingleAircraftDiscrete9HEREnv()
    M = 200
    ag = rng.uniform(0, 1, (M, 2)); g = ag + rng.uniform(-0.06, 0.06, (M, 2))
    g[:6] = ag[:6] + np.array([[20.0 / 800, 0.0]])
    r = np.array([env.compute_reward(ag[i].copy(), g[i].copy(), None) for i in range(M)], np.float64)
    ag_after = ag[0].copy(); env.compute_reward(ag_after, g[0].copy(), None)      # unnormalize_position works in place
    inputs = np.zeros((M, 26))
    for i in range(M):
        ob = env.reset()
        v = np.concatenate([ob["observation"], ob["desired_goal"]])
        if i % 3 == 0:       # put a listed intruder close to the ownship
            k = int(rng.randint(4))
            v[4 * k + 4: 4 * k + 6] = v[0:2] + rng.uniform(-0.03, 0.03, 2)
        if i % 5 == 1:       # goal next to the ownship
            v[-2:] = v[0:2] + rng.uniform(-0.03, 0.03, 2)
        inputs[i] = v
    ri = np.array([env.compute_input_reward(inputs[i].copy()) for i in range(M)], np.float64)
    np.savez_compressed(os.path.join(HERE, "d9her_reward.npz"), ag=ag, g=g, r=r, ag0_after=ag_after, inputs=inputs, ri=ri)
    return {"d9her_reward": {"pairs": M}}


def make_her_sampler_golden():
    """Outputs of the unmodified baselines sampler (her_sampler.py:19-61) on synthetic episode batches, with the four
    np.random draws recorded; reward_fun = compute_reward of the two GoalEnv variants of the package."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "ref_her_sampler", os.path.join(REF, "Algorithms", "baselines-master", "baselines", "her", "her_sampler.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    PkgConfig.intruder_size = 0
    np.random.seed(3)
    her, dher = SingleAircraftHEREnv(), SingleAircraftDiscreteHEREnv()
    rng = np.random.RandomState(11)
    out = {}
    for name, env, E, T, dim_o, batch, k, pix in (("her", her, 6, 12, 10, 256, 4, False), ("dher", dher, 9, 30, 18, 512, 4, True),
                                                  ("none", dher, 5, 7, 6, 64, 0, True)):
        scale = 800.0 if pix else 1.0
        ag = np.cumsum(rng.normal(0, 6.0 if pix else 0.008, (E, T + 1, 2)), axis=1) + rng.uniform(0.2, 0.8, (E, 1, 2)) * scale
        eb = {"o": rng.uniform(-1, 1, (E, T + 1, dim_o)), "u": rng.uniform(-1, 1, (E, T, 1 if pix else 2)),
              "g": np.repeat(rng.uniform(0.1, 0.9, (E, 1, 2)) * scale, T, axis=1), "ag": ag}
        eb2 = dict(eb); eb2["o_2"] = eb["o"][:, 1:, :]; eb2["ag_2"] = eb["ag"][:, 1:, :]      # replay_buffer.py:46-47
        fn = mod.make_sample_her_transitions("future" if k else "none", k,
                                             lambda ag_2, g, info, env=env: env.compute_reward(ag_2, g, info))
        calls = []
        orig = {n: getattr(np.random, n) for n in ("randint", "uniform")}

        def wrap(n):
            def f(*a, **kw):
                v = orig[n](*a, **kw)
                calls.append(np.array(v))
                return v
            return f
        for n in orig:
            setattr(np.random, n, wrap(n))
        try:
            np.random.seed(21)
            tr = fn(eb2, batch)
        finally:
            for n, f in orig.items():
                setattr(np.random, n, f)
        assert len(calls) == 4
        for key, v in eb.items():
            out["%s_ep_%s" % (name, key)] = v
        for key, v in zip(("episode_idxs", "t_samples", "u_her", "u_offset"), calls):
            out["%s_draw_%s" % (name, key)] = v
        for key in ("o", "u", "g", "ag", "o_2", "ag_2", "r"):
            out["%s_tr_%s" % (name, key)] = np.asarray(tr[key])
        out["%s_meta" % name] = np.array([k, batch, env.goal_radius, 2 if pix else 1], np.float64)
    np.savez_compressed(os.path.join(HERE, "her_sampler.npz"), **out)
    return {"her_sampler": {"cases": 3}}


def main():
    only = os.environ.get("GCA_GOLDEN_ONLY")
    if only:                                   # add traces of new variants without regenerating the others
        with open(os.path.join(HERE, "META.json")) as f:
            meta = json.load(f)
        meta.update(make_env_goldens())
        if "d9her" in only.split(","):
            meta.update(make_d9her_reward_golden())
        if "her_sampler" in only.split(","):
            meta.update(make_her_sampler_golden())
        if "stack" in only.split(","):
            meta.update(make_stack_frame_golden())
        if "mctsrnd_model" in only.split(","):
            meta.update(make_mctsrnd_model_goldens())
        with open(os.path.join(HERE, "META.json"), "w") as f:
            json.dump(meta, f, indent=1, sort_keys=True)
        return
    meta = {"numpy": np.__version__, "python": sys.version.split()[0]}
    try:
        from threadpoolctl import threadpool_info
        meta["threadpools"] = [{k: str(v) for k, v in d.items()} for d in threadpool_info()]
    except Exception as e:  # pragma: no cover
        meta["threadpools"] = str(e)
    meta.update(make_env_goldens())
    meta.update(make_mcts_goldens())
    meta.update(make_mctsrnd_model_goldens())
    meta.update(make_her_reward_golden())
    meta.update(make_d9her_reward_golden())
    meta.update(make_her_sampler_golden())
    meta.update(make_stack_frame_golden())
    with open(os.path.join(HERE, "META.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
