"""Shared helpers for the parity tests: golden loading and state plumbing."""
import os

import numpy as np

from gca_b200 import variants

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

STATE_KEYS = ("own_pos", "own_hs", "own_vel", "own_vel_is_f32", "goal", "no_conflict", "ep_steps", "ipos",
              "ipos_is_f64", "ivel", "iflag", "ihs")
GOLDEN_VARIANTS = {"env": "SingleAircraftEnv", "env2": "SingleAircraft2Env", "her": "SingleAircraftHEREnv",
                   "dher": "SingleAircraftDiscreteHEREnv", "mcts": "SingleAircraftMCTSEnv",
                   "d9her": "SingleAircraftDiscrete9HEREnv", "d3her": "SingleAircraftDiscrete3HEREnv",
                   "simenv": "SimSingleAircraftEnv", "rndenv": "SingleAircraftRandomEnv",
                   "mctsrnd": "SingleAircraftMCTSRandIntruderEnv", "stack": "SingleAircraftStackEnv"}
GOLDEN_N = (0, 1, 3, 80)
GOLDEN_N_BY_VARIANT = {"d9her": (5, 12, 80), "d3her": (5, 12, 80), "simenv": (3, 80), "rndenv": (3, 80),
                       "mctsrnd": (1, 3, 80), "stack": (0, 3, 80)}     # the nearest-n observation needs more than Config.n = 4 intruders
# every (variant key, N) with a recorded trace file
GOLDEN_CASES = [(vk, n) for vk in sorted(GOLDEN_VARIANTS) for n in GOLDEN_N_BY_VARIANT.get(vk, GOLDEN_N)]
GOAL_VARIANTS = ("her", "dher", "d9her", "d3her")          # dict observation: achieved / desired goal outputs


def config_class(variant_key):
    if variant_key in ("mcts", "d9her", "d3her", "simenv", "rndenv", "mctsrnd"):
        from Simulators.config import Config
    else:
        from gym_guidance_collision_avoidance_single.envs.config import Config
    return Config


def golden_config(variant_key):
    return variants.make_config(GOLDEN_VARIANTS[variant_key], config_class(variant_key))


def load_trace(variant_key, n):
    return np.load(os.path.join(GOLDEN, "trace_%s_n%d.npz" % (variant_key, n)))


def golden_state(g, prefix, sel=None):
    """Canonical state dict from golden arrays with the given prefix ('s0_', or 'sa_'/'sr_' + index)."""
    def get(k):
        a = g[prefix + k]
        return a if sel is None else a[sel]
    st = {
        "own_pos": get("own_pos").astype(np.float32),
        "own_hs": np.stack([get("own_heading"), get("own_speed")], -1).astype(np.float64),
        "own_vel": get("own_vel").astype(np.float64),
        "own_vel_is_f32": get("own_vel_is_f32").astype(np.uint8),
        "goal": get("goal").astype(np.float64),
        "no_conflict": get("no_conflict").astype(np.int32),
        "ep_steps": get("steps").astype(np.int32),
        "ipos": get("ipos").astype(np.float64),
        "ipos_is_f64": get("ipos_is_f64").astype(np.uint8),
        "ivel": get("ivel").astype(np.float32),
        "iflag": get("iflag").astype(np.uint8),
    }
    # intruder (heading, speed): state only of the variant whose intruders turn (recorded as zeros elsewhere; absent
    # from the trace files made before that variant existed)
    st["ihs"] = get("ihs").astype(np.float64) if prefix + "ihs" in g.files else np.zeros(st["ipos"].shape, np.float64)
    return {k: np.ascontiguousarray(v) for k, v in st.items()}


def assert_state_equal(got, want, what="", skip=("ep_steps",), rows=None):
    for k in STATE_KEYS:
        if k in skip:
            continue
        a, b = got[k], want[k]
        if rows is not None:
            a = a[rows]
        assert a.shape == b.shape, (what, k, a.shape, b.shape)
        if not np.array_equal(a, b):
            bad = np.argwhere(a != b)
            raise AssertionError("%s: state field %s differs at %s: got %r want %r" % (
                what, k, bad[:4].tolist(), a[tuple(bad[0])], b[tuple(bad[0])]))


class ShardedOracle(object):
    """The oracle over a whole batch, split into contiguous env ranges (bench.oracle_shards): one OracleEnv per host
    thread, each with the env_id0 of its first env, so every env draws what the device's env of that global id draws.
    ctypes releases the GIL, so the shards step in parallel.  Outputs and state are concatenated on demand."""

    def __init__(self, cfg, B, N, seed, env_id0=0, f32_positions=True):
        from concurrent.futures import ThreadPoolExecutor
        from oracle import oracle as orc
        threads = min(os.cpu_count() or 1, B)
        self.bounds = [(int(r[0]), int(r[-1]) + 1) for r in np.array_split(np.arange(B), threads)]
        self.shards = [orc.OracleEnv(cfg, hi - lo, N, draws=1, trig=orc.TRIG_SHARED, seed=seed, env_id0=env_id0 + lo,
                                     f32_positions=f32_positions, auto_reset=True) for lo, hi in self.bounds]
        self.pool = ThreadPoolExecutor(threads)
        self.cfg, self.B, self.N, self.D = cfg, B, N, self.shards[0].D

    def _each(self, fn):
        list(self.pool.map(fn, range(len(self.shards))))

    def reset(self):
        self._each(lambda i: self.shards[i].reset())
        return self.obs

    def step(self, actions):
        """actions: [B, 2] f64 (continuous) or [B] codes (discrete)."""
        self._each(lambda i: self.shards[i].step(actions[self.bounds[i][0]:self.bounds[i][1]]))

    def _cat(self, name):
        return np.concatenate([getattr(s, name) for s in self.shards])

    obs = property(lambda self: self._cat("obs"))
    reward = property(lambda self: self._cat("reward"))
    done = property(lambda self: self._cat("done"))
    info = property(lambda self: self._cat("info"))
    achieved = property(lambda self: self._cat("achieved"))
    desired = property(lambda self: self._cat("desired"))
    nearest = property(lambda self: self._cat("nearest"))

    @property
    def state(self):
        return {k: np.concatenate([s.state[k] for s in self.shards]) for k in self.shards[0].state}

    def close(self):
        self.pool.shutdown()


def golden_actions(variant_key, g):
    """[traces][T][2] action array of a golden file in the form the batched API takes:
    int codes in column 0 for the discrete kinds (the MCTS env's (a0, a1) tuple is a0*3+a1)."""
    a = np.array(g["actions"], np.float64)
    if variant_key in ("mcts", "mctsrnd"):
        a[..., 0] = a[..., 0] * 3 + a[..., 1]
        a[..., 1] = 0
    return a


# ------------------------------------------------------------------------------- fast (fp32) mode tolerance
# north star: "within a stated tolerance in an fp32 mode".  Stated here (and in DESIGN.md section 2), against the traces
# recorded from the unmodified reference, free running over the whole recorded horizon (25-40 steps, resets included):
#   flags (info / event code), done, no_conflict, per-intruder conflict flags, number of draws consumed: IDENTICAL
#   positions (pixels)                         |d| <= 2e-3   (measured 1.1e-3: a retried spawn is stored rounded to f32, Q3)
#   normalised observation entries, goals      |d| <= 3e-6   (measured 1.3e-6; outputs are f32: 6e-8 of that is the cast)
#   raw observation entries (pixels; MCTS envs) |d| <= 2e-3
#   reward                                     |d| <= 2e-7   (measured 6.3e-8; -d/1200 rounded to f32)
#   dist_nearest_intruder (Discrete3HER)       |d| <= 1e-3   (measured 2.7e-4)
FAST_TOL = {"pos": 2e-3, "obs": 3e-6, "obs_raw": 2e-3, "reward": 2e-7, "nearest": 1e-3}
RAW_OBS_VARIANTS = ("mcts", "mctsrnd")


def fast_obs_tol(variant_key):
    return FAST_TOL["obs_raw"] if variant_key in RAW_OBS_VARIANTS else FAST_TOL["obs"]
