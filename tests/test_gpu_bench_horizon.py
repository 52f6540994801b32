"""Every env workload of bench.py, run as bench.py runs it - its shapes, seeds, variants, action dtypes, warm-up counts,
CUDA graphs and replays, profiled and host-buffer steps, at its default --steps / --warmup - against the CPU oracle,
bit for bit, over the whole horizon.

Over that horizon every env goes through several episodes and its tick reaches the thousands, the ownship-record stamps
(and the tile walk direction they pick) are carried across thousands of graph replays, the dead position plane is
discarded on every step, and rare events (NMAC and map exit in one step, retried spawns, dense respawn lists) coincide
on their own.  A capture executes nothing, so the oracle steps for the steps that run: warm-up steps, replays x graph
length and eager steps.  Nothing is added to a captured graph; only the last step of a replay leaves its outputs, so
the outputs are compared at replay boundaries.  At every checkpoint: every output (reward and floats by their bits, so
-0.0 counts), the whole state with ticks and counters, the number of episodes every env finished, and gca_check (a
streaming lane that gave up waiting for its ownship record).  Each case asserts that it reached what it is there for.

bench_mcts and bench_her_replay are not here: tests/test_gpu_bench_shapes.py checks both at their bench sizes."""
import time

import numpy as np
import pytest

import bench
from helpers import ShardedOracle
from test_gpu_bench_shapes import _sample
from test_gpu_raster_paths import _oracle_frames

pytestmark = pytest.mark.gpu

NMAC, CONFLICT, GOAL, WALL = 1, 2, 3, 4


def _bench_defaults():
    """bench.py's default --steps and --warmup: what main() hands to main_gpu for an empty command line."""
    import sys
    import unittest.mock as um
    args = {}
    with um.patch.object(sys, "argv", ["bench.py"]), um.patch.object(bench, "main_gpu", lambda a: args.update(vars(a))):
        bench.main()
    return args["steps"], args["warmup"]


def _torch():
    import torch
    return torch


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.itemsize == 4 else np.uint64) if a.dtype.kind == "f" else a


def _same(got, want, what):
    g, w = _bits(got), _bits(want)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    if not np.array_equal(g, w):
        bad = np.argwhere(g != w)
        raise AssertionError("%s: %d entries differ, first at %s: got %r want %r" % (
            what, len(bad), bad[:4].tolist(), got[tuple(bad[0])], want[tuple(bad[0])]))


def _host_actions(a):
    """What the oracle takes for a device action batch: f64 (an f32 batch is exact in f64), or the int codes."""
    a = a.cpu().numpy()
    return a.astype(np.float64) if a.dtype.kind == "f" else a.astype(np.int64)


class Horizon(object):
    """A device handle and its sharded oracle twin, with what the oracle saw on the way: events and finished episodes
    of every step, and the events and done rows of the steps whose outputs were compared."""

    def __init__(self, env, seed, env_id0=0):
        from gca_b200 import abi
        self.env = env
        fast = env.mode == abi.MODE_FAST
        self.ref = ShardedOracle(env.cfg, env.num_envs, env.n_intruders, seed, env_id0, f32_positions=fast)
        self.cast = (lambda x: x.astype(np.float32)) if fast else (lambda x: x)
        self.episodes = np.zeros(env.num_envs, np.int64)
        self.events = np.zeros(6, np.int64)          # every executed step
        self.seen = np.zeros(6, np.int64)            # the compared steps
        self.steps = self.checkpoints = self.done_checkpoints = 0
        self.t0 = time.perf_counter()

    def reset(self):
        got = self.env.reset().cpu().numpy()
        want = self.ref.reset()
        if self.ref.D:
            _same(got[:, :self.ref.D], self.cast(want), "reset obs")

    def step(self, host_actions):
        self.ref.step(host_actions)
        done = self.ref.done
        self.episodes += done
        self.events += np.bincount(self.ref.info, minlength=6)
        self.steps += 1

    def _each_shard(self, pairs):
        """pairs: (name, got [B, ...], shard -> want); compared shard by shard on the oracle's threads."""
        ref = self.ref

        def one(i):
            lo, hi = ref.bounds[i]
            return [np.array_equal(_bits(g[lo:hi]), _bits(w(ref.shards[i]))) for _, g, w in pairs]
        ok = np.array(list(ref.pool.map(one, range(len(ref.shards)))))
        return [name for (name, _, _), good in zip(pairs, ok.all(0)) if not good]

    def check(self, what, outs=None, state=True):
        """outs: host arrays of the outputs (default: the handle's device tensors).  state: also the whole state, the
        counters and gca_check (only when no step is in flight)."""
        env, ref, cast = self.env, self.ref, self.cast
        if outs is None:
            outs = {k: getattr(env, k).cpu().numpy() for k in ("obs", "reward", "done", "info")}
            if env.is_goal_env:
                outs.update(achieved=env.achieved.cpu().numpy(), desired=env.desired.cpu().numpy())
            if env.nearest is not None:
                outs["nearest"] = env.nearest.cpu().numpy()
        D = ref.D
        pairs = [("info", outs["info"], lambda s: s.info), ("done", outs["done"], lambda s: s.done),
                 ("reward", outs["reward"], lambda s: cast(s.reward))]
        if D:
            pairs.append(("obs", outs["obs"][:, :D], lambda s: cast(s.obs)))
        for k in ("achieved", "desired", "nearest"):
            if k in outs:
                pairs.append((k, outs[k], lambda s, k=k: cast(getattr(s, k))))
        st = None
        if state:
            st = env.get_state()                     # (synchronises and raises what gca_check reports)
            env.check()
            pairs += [(k, st[k], lambda s, k=k: s.state[k]) for k in st]
            counters = env.counters().cpu().numpy()
        bad = self._each_shard(pairs)
        if bad:                                      # the whole arrays, for the first index that differs
            want = {"info": ref.info, "done": ref.done, "reward": cast(ref.reward), "obs": cast(ref.obs),
                    "achieved": cast(ref.achieved), "desired": cast(ref.desired), "nearest": cast(ref.nearest)}
            for name, got, _ in pairs:
                if name in bad:
                    _same(got, want[name] if name in want else ref.state[name], "%s: %s" % (what, name))
        if state:
            _same(counters[:, 3], self.episodes.astype(np.int32), "%s: finished episodes" % (what,))
        done = outs["done"]
        self.seen += np.bincount(outs["info"], minlength=6)
        self.done_checkpoints += bool(done.any())
        self.checkpoints += 1
        return st

    def report(self, name):
        print("\n[%s] %d steps x %d envs = %.3g env-steps compared at %d checkpoints (%d with done rows); events of every "
              "step: nmac %d conflict %d goal %d wall %d; at checkpoints: nmac %d conflict %d goal %d wall %d; episodes "
              "finished: %d (max %d per env); %.0f s" % (
                  name, self.steps, self.env.num_envs, float(self.steps) * self.env.num_envs, self.checkpoints,
                  self.done_checkpoints, self.events[NMAC], self.events[CONFLICT], self.events[GOAL], self.events[WALL],
                  self.seen[NMAC], self.seen[CONFLICT], self.seen[GOAL], self.seen[WALL], self.episodes.sum(),
                  self.episodes.max(), time.perf_counter() - self.t0), flush=True)

    def assert_reached(self, steps, events=(NMAC, CONFLICT, GOAL, WALL), done_checkpoints=3):
        """events: the info codes the variant can end a step with (WALL: only the variants whose wall ends the episode;
        NMAC and CONFLICT: only with intruders)."""
        assert self.steps == steps, (self.steps, steps)
        assert np.all(self.ref.state["tick"] == 1 + steps)          # one tick for the reset, one per step
        for e in events:
            assert self.seen[e] > 0, ("event %d never compared" % e, self.seen)
        assert self.done_checkpoints >= done_checkpoints, self.done_checkpoints

    def close(self):
        self.env.close()
        self.ref.close()


def _graph_replays(h, step_fn, twin_fn, n_batches, reps=6):
    """bench.graph_step_ms call for call (3 warm-up steps on a side stream, a capture of n_batches steps, one replay,
    `reps` more), the oracle stepped for every step that runs, a check after the warm-up and after every replay.
    step_fn(i) may return a device tensor and twin_fn(i) the oracle's value of it; the values of a replay's steps are
    compared after it (the capture keeps every step's output tensor)."""
    torch = _torch()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(3):
            step_fn(i % n_batches)
            twin_fn(i % n_batches)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    h.check("graph warm-up")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = [step_fn(i) for i in range(n_batches)]
    for r in range(1 + reps):
        graph.replay()
        wants = [twin_fn(i) for i in range(n_batches)]           # (the oracle runs while the replay does)
        torch.cuda.synchronize()
        h.check("replay %d" % r)
        for i, (got, want) in enumerate(zip(outs, wants)):
            if want is not None:
                _same(got.cpu().numpy(), want, "replay %d, captured step %d" % (r, i))
    return 3 + (1 + reps) * n_batches


def _env(variant, B, cfg_cls, N, mode, seed, env_id0=0):
    from gca_b200.batched import BatchedAircraftEnv
    return BatchedAircraftEnv(variant, B, cfg_cls, n_intruders=N, mode=mode, draws="philox", seed=seed, env_id0=env_id0)


# ------------------------------------------------------------------------------------------------ the headline
def _headline(rank, replays=None):
    """bench.main_gpu on rank `rank`: warm-up, the timed replays (+ eager remainder), the profiled eager steps and both
    host-buffer paths.  replays=None: as many as bench's default --steps makes, and everything after them."""
    torch = _torch()
    from gym_guidance_collision_avoidance_single.envs.config import Config
    K, W = _bench_defaults()
    W = max(W, 3)
    B, N, GS = bench.ENVS_PER_GPU, bench.N_INTRUDERS, bench.GRAPH_STEPS
    env = _env(bench.VARIANT, B, Config, N, "fast", seed=2024, env_id0=rank * B)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1 + rank)
    actions = [torch.rand((B, 2), device="cuda", generator=gen) * 2 - 1 for _ in range(GS)]
    host = [_host_actions(a) for a in actions]
    h = Horizon(env, seed=2024, env_id0=rank * B)
    h.reset()
    torch.cuda.synchronize()

    G = max(1, min(K, GS))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(W):
            env.step(actions[i % GS])
            h.step(host[i % GS])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    h.check("after warm-up")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(G):
            env.step(actions[i])
    full = replays is None
    replays = K // G if full else replays
    for r in range(1 + replays):                      # the untimed replay, then the timed ones
        graph.replay()
        for i in range(G):
            h.step(host[i])
        torch.cuda.synchronize()
        h.check("replay %d" % r)
    if not full:
        h.report("headline rank %d" % rank)
        h.assert_reached(W + (1 + replays) * G)
        h.close()
        return
    for i in range(K - replays * G):                  # bench's eager remainder (none at the default --steps)
        env.step(actions[i])
        h.step(host[i])
    if K % G:
        torch.cuda.synchronize()
        h.check("eager remainder")

    Kp = max(20, min(K, 200))                         # profiled eager steps: events between the kernels
    env.profile(True)
    for i in range(Kp):
        env.step(actions[i % GS])
        h.step(host[i % GS])
        if (i + 1) % 50 == 0 or i + 1 == Kp:
            h.check("profiled step %d" % i)
    prof = env.read_profile()
    env.profile(False)
    assert prof["steps"] == Kp and prof["intruders_ms"] > 0, prof

    host_actions = [a.cpu().numpy() for a in actions[:8]]
    Ke = max(3, min(K, 300))
    # (bench binds its thread to the GPU's NUMA node here; that places the pinned buffers, it changes no result)
    for i in range(3):
        outs = env.step_host(host_actions[i % 8])
        h.step(host_actions[i % 8].astype(np.float64))
        h.check("step_host warm-up %d" % i, dict(zip(("obs", "reward", "done", "info"), outs)))
    for i in range(Ke):                               # (a) one step at a time
        obs, rew, dn, info = env.step_host(host_actions[i % 8])
        h.step(host_actions[i % 8].astype(np.float64))
        h.check("step_host %d" % i, {"obs": obs, "reward": rew, "done": dn, "info": info})
    for i in range(2):                                # (b) begin / wait, two steps in flight
        env.step_host_begin(host_actions[i % 8])
        outs = env.step_host_wait()
        h.step(host_actions[i % 8].astype(np.float64))
        h.check("step_host_begin warm-up %d" % i, dict(zip(("obs", "reward", "done", "info"), outs)))
    env.step_host_begin(host_actions[0])
    prev = 0
    for i in range(1, Ke):
        env.step_host_begin(host_actions[i % 8])
        obs, rew, dn, info = env.step_host_wait()     # the step begun before; step i is in flight: outputs only
        h.step(host_actions[prev % 8].astype(np.float64))
        h.check("step_host_wait %d" % (i - 1), {"obs": obs, "reward": rew, "done": dn, "info": info}, state=False)
        prev = i
    obs, rew, dn, info = env.step_host_wait()
    h.step(host_actions[prev % 8].astype(np.float64))
    torch.cuda.synchronize()
    h.check("step_host_wait %d" % prev, {"obs": obs, "reward": rew, "done": dn, "info": info})
    env.check()
    h.report("headline rank %d" % rank)
    h.assert_reached(W + (1 + K // G) * G + K % G + Kp + 3 + Ke + 2 + Ke)
    assert (h.episodes >= 1).mean() >= 0.5 and h.episodes.max() >= 3, np.bincount(h.episodes)
    h.close()


def test_headline_rank0_whole_bench_sequence_vs_oracle():
    """bench.main_gpu on one GPU: 20 warm-up steps on a side stream, 1 + 40 replays of a 50-step graph, 200 profiled
    eager steps, 3 + 300 step_host and 2 + 300 step_host_begin / _wait steps; actions: bench's 50 torch.rand batches of
    generator seed 1 (f32, exact in the oracle's f64), the first 8 of them from host memory."""
    _headline(0)


def test_headline_rank7_env_ids_vs_oracle():
    """Rank 7 of an 8-GPU torchrun: env ids 7 x 65,536 onward, action generator seed 8; the warm-up, the untimed replay
    and 10 timed replays."""
    _headline(7, replays=10)


# ------------------------------------------------------------------------------------------------ the other legs
def test_her_leg_with_relabel_rewards_vs_oracle():
    """bench_her: SingleAircraftHEREnv, 5 + 200 eager steps then an 8-step graph, each step followed by
    compute_reward(achieved [B, 2], goals [4, B, 2]); every relabel reward by its bits (the HER kind's 0 is -0.0)."""
    torch = _torch()
    from gca_b200 import abi
    from gca_b200.batched import compute_reward
    from gym_guidance_collision_avoidance_single.envs.config import Config
    from oracle import oracle as orc
    torch.manual_seed(4)
    B, N, k = bench.ENVS_PER_GPU, bench.N_INTRUDERS, 4
    env = _env("SingleAircraftHEREnv", B, Config, N, "fast", seed=4)
    h = Horizon(env, seed=4)
    h.reset()
    acts = [torch.rand((B, 2), device="cuda") * 2 - 1 for _ in range(8)]
    goals = torch.rand((k, B, 2), device="cuda")
    host, goals_h = [_host_actions(a) for a in acts], goals.cpu().numpy()
    relabels = [0]

    def one(i):
        env.step(acts[i % 8])
        return compute_reward(env.achieved, goals, Config.goal_radius, abi.OBS_HER)

    def twin(i):
        h.step(host[i % 8])
        ag = np.broadcast_to(h.ref.achieved.astype(np.float32), goals_h.shape)
        relabels[0] += goals_h.shape[0] * goals_h.shape[1]
        return orc.compute_reward(ag, goals_h, Config.goal_radius, abi.OBS_HER)
    for n, i in enumerate(list(range(5)) + list(range(200))):          # 5 warm-up calls, then 200 timed ones
        got = one(i)
        want = twin(i)
        if n == 4 or (n - 4) % 50 == 0:
            h.check("eager step %d" % n)
            _same(got.cpu().numpy(), want, "eager step %d relabel rewards" % n)
    steps = 5 + 200 + _graph_replays(h, one, twin, 8)
    h.report("her")
    print("[her] %d relabel rewards computed, those of %d steps compared" % (relabels[0], 5 + 8 * 7), flush=True)
    h.assert_reached(steps, events=(NMAC, CONFLICT, GOAL))
    h.close()


def _discrete_leg(name, variant, seed, n_actions, eager_acts=0, torch_seed=0):
    """bench_d9her / its d3her half / bench_mctsrnd's env part / bench_n0: `eager_acts` batches of int32 actions for
    5 eager steps (+ 200 timed ones when there are 8 of them), then a graph of GRAPH_STEPS steps."""
    torch = _torch()
    from Simulators.config import Config as SimConfig
    torch.manual_seed(torch_seed)
    B, N, GS = bench.ENVS_PER_GPU, bench.N_INTRUDERS, bench.GRAPH_STEPS
    env = _env(variant, B, SimConfig, N, "fast", seed=seed)
    h = Horizon(env, seed=seed)
    h.reset()
    steps = 0
    if eager_acts:
        acts = [torch.randint(0, n_actions, (B,), device="cuda", dtype=torch.int32) for _ in range(eager_acts)]
        host = [_host_actions(a) for a in acts]
        eager = list(range(5)) + (list(range(200)) if eager_acts == 8 else [])   # warm-up calls, then timed ones
        for n, i in enumerate(eager):
            env.step(acts[i % eager_acts])
            h.step(host[i % eager_acts])
            if n == 4 or (n - 4) % 50 == 0:
                h.check("eager step %d" % n)
        steps += len(eager)
    acts50 = acts if eager_acts == GS else \
        [torch.randint(0, n_actions, (B,), device="cuda", dtype=torch.int32) for _ in range(GS)]
    host50 = [_host_actions(a) for a in acts50]
    steps += _graph_replays(h, lambda i: env.step(acts50[i]), lambda i: h.step(host50[i]), GS)
    h.report(name)
    return h, steps


def test_d9her_leg_vs_oracle():
    """bench_d9her: SingleAircraftDiscrete9HEREnv (nearest-4 observation, dict goals), 5 + 200 eager steps over 8
    action batches, then a graph of 50."""
    h, steps = _discrete_leg("d9her", "SingleAircraftDiscrete9HEREnv", 6, 9, eager_acts=8, torch_seed=6)
    h.assert_reached(steps, events=(NMAC, CONFLICT, GOAL))
    h.close()


def test_d3her_leg_vs_oracle():
    """bench_d9her's Discrete(3) sibling: the nearest-intruder distance output too; a graph of 50."""
    h, steps = _discrete_leg("d3her", "SingleAircraftDiscrete3HEREnv", 7, 3, torch_seed=7)
    assert h.env.nearest is not None
    h.assert_reached(steps, events=(NMAC, CONFLICT, GOAL))
    h.close()


def test_mctsrnd_leg_and_planner_model_vs_oracle():
    """bench_mctsrnd: SingleAircraftMCTSRandIntruderEnv, 5 eager steps and a graph of 50 on the same 50 action batches;
    then the random-intruder planner model (100 playouts of depth 3) on the first 2,048 observations as f64 roots,
    seeds 1 .. 11, a seeded sample of 256 roots of every launch replayed by the oracle under its own root id."""
    torch = _torch()
    from gca_b200 import abi, mcts
    from Algorithms.MCTS.config_single import Config as MctsConfig
    from oracle import oracle as orc
    h, steps = _discrete_leg("mctsrnd", "SingleAircraftMCTSRandIntruderEnv", 8, 9, eager_acts=bench.GRAPH_STEPS,
                             torch_seed=8)
    h.assert_reached(steps, events=(NMAC, CONFLICT, GOAL))
    env, N = h.env, h.env.n_intruders
    R, P, depth = 2048, 100, 3
    roots = env.obs[:R].double().contiguous()
    _same(roots.cpu().numpy(), h.ref.obs[:R].astype(np.float32).astype(np.float64), "roots")
    host = roots.cpu().numpy()
    mcfg = abi.make_mcts_config(MctsConfig, random_intruders=True)
    launches = [mcts.playouts(roots, P, depth=depth, cfg=mcfg, seed=1)]
    torch.cuda.synchronize()
    for rep_i in range(10):
        launches.append(mcts.playouts(roots, P, depth=depth, cfg=mcfg, seed=2 + rep_i))
    torch.cuda.synchronize()
    flags = []
    for s, (rw, first, fl) in enumerate(launches, start=1):
        rw, first, fl = rw.cpu().numpy(), first.cpu().numpy(), fl.cpu().numpy()
        rows = _sample(R, 100 + s)
        want = list(h.ref.pool.map(lambda r: orc.mcts_playouts(mcfg, N, host[r:r + 1], P, depth, seed=s,
                                                               root_id0=int(r)), rows))
        for r, (wr, wf, wfl) in zip(rows, want):
            what = "seed %d root %d" % (s, r)
            _same(fl[r], wfl[0], what + " flags")
            _same(first[r], wf[0], what + " first actions")
            _same(rw[r], wr[0], what + " rewards")
        flags.append(fl[rows])
    fl = np.concatenate(flags)
    print("[mctsrnd model] %d launches x 256 roots x %d playouts compared; terminal %.2f, wall %.2f, conflict %.2f, "
          "roots with every playout terminal %.2f" % (len(launches), P, (fl != 0).mean(), ((fl & abi.MCTS_WALL) != 0).mean(),
                                                      ((fl & abi.MCTS_CONFLICT) != 0).mean(), (fl != 0).all(1).mean()))
    assert (fl & abi.MCTS_WALL).any() and (fl & abi.MCTS_CONFLICT).any() and (fl != 0).all(1).any()
    h.close()


def test_faithful_leg_vs_oracle():
    """bench_faithful: the headline variant in FAITHFUL mode (f64 observations, f32 / f64 positions), f64 actions, a
    graph of 50."""
    torch = _torch()
    from gym_guidance_collision_avoidance_single.envs.config import Config
    torch.manual_seed(9)
    B, N, GS = bench.ENVS_PER_GPU, bench.N_INTRUDERS, bench.GRAPH_STEPS
    env = _env(bench.VARIANT, B, Config, N, "faithful", seed=9)
    h = Horizon(env, seed=9)
    h.reset()
    acts = [torch.rand((B, 2), device="cuda", dtype=torch.float64) * 2 - 1 for _ in range(GS)]
    host = [_host_actions(a) for a in acts]
    steps = _graph_replays(h, lambda i: env.step(acts[i]), lambda i: h.step(host[i]), GS)
    h.report("faithful")
    h.assert_reached(steps)
    h.close()


def test_n0_leg_both_batches_vs_oracle():
    """bench_n0: SingleAircraftEnv without intruders (the one-kernel step), 65,536 and 4 Mi envs, a graph of 50 each."""
    torch = _torch()
    from gym_guidance_collision_avoidance_single.envs.config import Config
    torch.manual_seed(8)
    GS = bench.GRAPH_STEPS
    for B in (bench.ENVS_PER_GPU, 4 * 1024 * 1024):
        env = _env("SingleAircraftEnv", B, Config, 0, "fast", seed=8)
        h = Horizon(env, seed=8)
        h.reset()
        acts = [torch.randint(0, 9, (B,), device="cuda", dtype=torch.int32) for _ in range(GS)]
        host = [_host_actions(a) for a in acts]
        steps = _graph_replays(h, lambda i: env.step(acts[i]), lambda i: h.step(host[i]), GS)
        h.report("n0 %d envs" % B)
        h.assert_reached(steps, events=(GOAL,))
        h.close()


def test_stack_leg_frames_vs_oracle():
    """bench_stack: ImageBatch at 65,536 x 80 with a 4-frame ring, 3 + 10 eager steps; the whole state after every
    step, every plane of the ring of a seeded sample of 512 envs against VecFrameStack made of oracle frames, and the
    stack of every env that finished at the step."""
    torch = _torch()
    from gca_b200.stack import ImageBatch
    from gym_guidance_collision_avoidance_single.envs.config import Config
    torch.manual_seed(3)
    B, N, k = bench.ENVS_PER_GPU, bench.N_INTRUDERS, 4
    env = ImageBatch(B, Config, n_intruders=N, frame_stack=k, device=0, seed=3)
    h = Horizon(env.batch, seed=3)
    env.reset()
    h.ref.reset()
    sp = env.sprites.cpu().numpy()
    rows = np.sort(np.random.RandomState(512).choice(B, 512, replace=False))
    rows_d = torch.as_tensor(rows, device="cuda")

    def ring_rows():                                  # [512, k, H, W], oldest plane first
        return env.ring[rows_d][:, env.plane_order()].cpu().numpy()
    model = np.zeros((len(rows), k, env.H, env.W), np.uint8)
    model[:, -1] = _oracle_frames(Config, h.check("reset"), rows, sp)
    _same(ring_rows(), model, "ring after reset")
    acts = [torch.randint(0, 9, (B,), device="cuda", dtype=torch.int32) for _ in range(4)]
    host = [_host_actions(a) for a in acts]
    finished = 0
    for i in range(3 + 10):
        env.step(acts[i % 4])
        h.step(host[i % 4])
        st = h.check("step %d" % i)
        d = h.ref.done.astype(bool)
        model = np.roll(model, -1, axis=1)            # vec_frame_stack.py:17-24
        model[d[rows]] = 0
        model[:, -1] = _oracle_frames(Config, st, rows, sp)
        _same(ring_rows(), model, "ring after step %d" % i)
        fin = np.nonzero(d)[0]                        # every env that finished: an all-zero stack under the new frame
        if len(fin):
            got = env.ring[torch.as_tensor(fin, device="cuda")][:, env.plane_order()].cpu().numpy()
            assert not got[:, :-1].any(), ("older planes of finished envs after step %d" % i, fin[:4].tolist())
            _same(got[:, -1], _oracle_frames(Config, st, fin, sp), "newest frame of finished envs after step %d" % i)
        finished += len(fin)
    h.report("stack")
    print("[stack] frames of %d finished envs compared" % finished, flush=True)
    h.assert_reached(13, events=(GOAL,))
    assert finished > 0
    h.close()
