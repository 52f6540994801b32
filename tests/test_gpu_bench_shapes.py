"""The workloads of bench.py at bench.py's sizes and in its launch mode: a step captured in a CUDA graph and replayed
equals the same steps launched eagerly (and the oracle), the HER sampler and compute_reward past their first
grid-stride pass, and the MCTS kernels on bench-sized root batches (large per-root workspace offsets), each checked
bit for bit against the CPU oracle on a seeded sample of rows."""
import numpy as np
import pytest

from helpers import assert_state_equal, config_class, golden_config

pytestmark = pytest.mark.gpu


def _torch():
    import torch
    return torch


# ------------------------------------------------------------------------------------------------ graph replay
def _capture(env, step_fn, warmup, G):
    """bench.py's protocol: warm-up steps on a side stream, then torch.cuda.graph over G steps."""
    torch = _torch()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(warmup):
            step_fn(i % G)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    outs = []
    with torch.cuda.graph(graph):
        for i in range(G):
            outs.append(step_fn(i))
    return graph, outs


def _make(vk, B, N, seed):
    from gca_b200.batched import BatchedAircraftEnv
    from helpers import GOLDEN_VARIANTS
    return BatchedAircraftEnv(GOLDEN_VARIANTS[vk], B, config_class(vk), n_intruders=N, mode="fast", draws="philox",
                              seed=seed)


def _acts(env, G, seed):
    torch = _torch()
    g = torch.Generator(device="cuda").manual_seed(seed)
    B = env.num_envs
    if env.continuous:
        return [torch.rand((B, 2), device="cuda", generator=g) * 2 - 1 for _ in range(G)]     # float32: no conversion
    return [torch.randint(0, 9, (B,), device="cuda", dtype=torch.int32, generator=g) for _ in range(G)]


def _host(env):
    return [x.cpu().numpy().copy() for x in (env.obs, env.reward, env.done, env.info, env.achieved, env.desired)]


@pytest.mark.parametrize("vk,G", [("env2", 50), ("env2", 7), ("d9her", 50), ("d9her", 7), ("her", 8)])
def test_graph_replay_equals_eager_at_bench_size(vk, G):
    """65,536 envs x 80 intruders, FAST, Philox, auto-reset: the captured handle replayed R times against a twin handle
    stepped eagerly with the same actions; an odd G leaves the position plane flipped between replays.  her: bench_her's
    chain, the step followed by compute_reward([B, 2] vs [k, B, 2]) inside the capture."""
    torch = _torch()
    from gca_b200 import abi
    from gca_b200.batched import compute_reward
    B, N, W, R = 65536, 80, 3, 3
    cap, eag = _make(vk, B, N, seed=2024), _make(vk, B, N, seed=2024)
    acts = _acts(cap, G, seed=1)
    goals = torch.rand((4, B, 2), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    radius = config_class(vk).goal_radius

    def stepper(env):
        def one(i):
            env.step(acts[i])
            return compute_reward(env.achieved, goals, radius, abi.OBS_HER) if vk == "her" else None
        return one
    cap.reset()
    eag.reset()
    graph, outs = _capture(cap, stepper(cap), W, G)
    eager = stepper(eag)
    for i in range(W):
        eager(i % G)
    for rep in range(R):
        graph.replay()
        torch.cuda.synchronize()
        want_rewards = [eager(i) for i in range(G)]
        for a, b in zip(_host(cap), _host(eag)):
            assert np.array_equal(a, b), (vk, G, rep)
        if vk == "her":
            for i in range(G):
                assert torch.equal(outs[i], want_rewards[i]), (rep, i)
                assert torch.equal(torch.signbit(outs[i]), torch.signbit(want_rewards[i]))
    sc, se = cap.get_state(), eag.get_state()
    assert_state_equal(sc, se, "graph vs eager", skip=())
    assert np.array_equal(sc["tick"], se["tick"])
    cap.close()
    eag.close()


@pytest.mark.parametrize("vk,G", [("env2", 7), ("d9her", 8)])
def test_graph_replay_ragged_vs_oracle(vk, G):
    torch = _torch()
    from oracle import oracle as orc
    B, N, W, R = 1000, 80, 3, 3
    env = _make(vk, B, N, seed=77)
    ref = orc.OracleEnv(golden_config(vk), B, N, draws=1, trig=orc.TRIG_SHARED, seed=77, f32_positions=True,
                        auto_reset=True)
    acts = _acts(env, G, seed=3)
    host_acts = []
    for a in acts:
        h = a.cpu().numpy().astype(np.float64)
        host_acts.append(h if env.continuous else np.stack([h, np.zeros(B)], -1))
    assert np.array_equal(env.reset().cpu().numpy(), ref.reset().astype(np.float32))
    graph, _ = _capture(env, lambda i: env.step(acts[i]), W, G)
    for i in range(W):
        ref.step(host_acts[i % G])
    for rep in range(R):
        graph.replay()
        torch.cuda.synchronize()
        for i in range(G):
            ref.step(host_acts[i])
        assert np.array_equal(env.obs.cpu().numpy(), ref.obs.astype(np.float32)), rep
        assert np.array_equal(env.reward.cpu().numpy(), ref.reward.astype(np.float32)), rep
        assert np.array_equal(env.done.cpu().numpy(), ref.done) and np.array_equal(env.info.cpu().numpy(), ref.info)
    assert_state_equal(env.get_state(), ref.state, "final state", skip=())
    env.close()


# ------------------------------------------------------------------------------------------------ HER sampler
def _episodes(E, T, dim_o, dim_u, dtype, seed):
    rng = np.random.RandomState(seed)
    eb = {"o": np.random.default_rng(seed).random((E, T + 1, dim_o), dtype=np.float32), "u": rng.uniform(-1, 1, (E, T, dim_u)),
          "g": rng.uniform(100, 700, (E, T, 2)),
          "ag": np.cumsum(rng.normal(0, 7, (E, T + 1, 2)), 1) + rng.uniform(100, 700, (E, 1, 2))}
    return {k: v.astype(dtype) for k, v in eb.items()}


@pytest.mark.parametrize("E,dim_o,batch,dtype", [(4096, 326, 262144, "float32"), (512, 326, 100003, "float64"),
                                                 (64, 27, 37888, "float32"), (64, 27, 37889, "float32")])
def test_her_sampler_past_one_pass_vs_oracle(E, dim_o, batch, dtype):
    """bench_her_replay's shape (E = 4096, T = 50, dim_o = 326, 262,144 transitions: 7 grid-stride passes of 37,888),
    an f64 buffer, and batches of exactly one pass and one more."""
    torch = _torch()
    from gca_b200 import replay
    from oracle import her_sampler as ohs
    T, k, radius, kind = 50, 4, 20.0, ohs.OBS_HER
    eb = _episodes(E, T, dim_o, 2, dtype, seed=E + batch)
    draws = ohs.philox_draws(batch, E, T, seed=99, call=3)
    want, ft = ohs.sample_her_transitions(eb, batch, k, radius, kind, draws)
    if dtype == "float32":                      # the device compares the f32 norm with the f32 radius
        d = np.sqrt(((want["ag_2"] - want["g"]) ** 2).sum(-1, dtype=np.float32), dtype=np.float32)
        want["r"] = -(d > np.float32(radius)).astype(np.float32)
    dev = {key: torch.as_tensor(v, device="cuda") for key, v in eb.items()}
    got, drawn = replay.sample_her_transitions(dev, batch, k, radius, kind, seed=99, call=3, return_draws=True)
    assert np.array_equal(drawn["episode"].cpu().numpy(), draws["episode_idxs"])
    assert np.array_equal(drawn["t"].cpu().numpy(), draws["t_samples"])
    assert np.array_equal(drawn["future_t"].cpu().numpy(), ft)
    for key in ("o", "u", "g", "ag", "o_2", "ag_2"):
        assert np.array_equal(got[key].cpu().numpy(), want[key]), key
    r = got["r"].cpu().numpy()
    assert np.array_equal(r.view(np.uint32), want["r"].view(np.uint32))        # the HER kind's 0 is -0.0
    assert np.all(np.signbit(r)) and (r == 0).any() and (r == -1).any()


# ------------------------------------------------------------------------------------------------ compute_reward
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("n_ag,k", [(1 << 18, 4), (151553, 5), (4 << 18, 1), (700001, 1)])
def test_compute_reward_past_one_pass_vs_oracle(n_ag, k, dtype):
    """Plain (k = 1) and tiled ([n_ag, 2] against [k, n_ag, 2]) forms past the 606,208 pairs of one grid-stride pass,
    with pairs at exactly goal_radius (12-16-20 offsets): `>` and `<` are strict; the HER kind returns -0.0."""
    torch = _torch()
    from gca_b200 import abi
    from gca_b200.batched import compute_reward
    from oracle import oracle as orc
    rng = np.random.RandomState(n_ag + k)
    ag = np.round(rng.uniform(0, 800, (n_ag, 2)))
    g = ag[None] + rng.uniform(-30, 30, (k, n_ag, 2))
    edge = rng.rand(k, n_ag) < 0.25
    sgn = rng.choice([-1.0, 1.0], (k, n_ag, 2))
    swap = rng.rand(k, n_ag) < 0.5
    off = np.where(swap[..., None], [16.0, 12.0], [12.0, 16.0]) * sgn
    g[edge] = (ag[None] + off)[edge]
    ag, g = ag.astype(dtype), g.astype(dtype)
    dev = lambda x: torch.as_tensor(np.ascontiguousarray(x), device="cuda")
    for kind in (abi.OBS_HER, abi.OBS_DHER):
        want = orc.compute_reward(np.broadcast_to(ag, g.shape).reshape(-1, 2), g.reshape(-1, 2), 20.0, kind).reshape(k, n_ag)
        got = compute_reward(dev(ag), dev(g if k > 1 else g[0]), 20.0, kind).cpu().numpy().reshape(k, n_ag)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), kind
        late = np.zeros((k, n_ag), bool)
        late.reshape(-1)[606208:] = True
        assert (edge & late).any() and (got[edge] == (0.0 if kind == abi.OBS_DHER else -0.0)).all()
        if kind == abi.OBS_HER:
            assert np.all(np.signbit(got)) and (got == 0).any() and (got == -1).any()


# ------------------------------------------------------------------------------------------------ MCTS
def _mcts_roots(R, seed, random_intruders=False):
    from gca_b200.batched import BatchedAircraftEnv
    from Simulators.config import Config as SimConfig
    if random_intruders:    # bench_mctsrnd: f32 observations of the random-intruder env, as f64 roots
        env = BatchedAircraftEnv("SingleAircraftMCTSRandIntruderEnv", R, SimConfig, n_intruders=80, mode="fast",
                                 draws="philox", seed=seed)
        env.reset()
        roots = env.obs.double().contiguous().clone()
    else:
        env = BatchedAircraftEnv("SingleAircraftMCTSEnv", R, SimConfig, n_intruders=80, mode="faithful", seed=seed)
        roots = env.reset().clone()
    env.close()
    return roots


def _sample(R, seed, m=256):
    rng = np.random.RandomState(seed)
    return np.sort(np.concatenate([[0, R - 1], rng.choice(np.arange(1, R - 1), m - 2, replace=False)]))


def test_mcts_search_bench_size_sampled_vs_oracle():
    """bench_mcts: gca_mcts_search on 65,536 roots (100 simulations, depth 3, N = 80), a seeded sample of 256 roots
    replayed by the oracle with their own root ids."""
    from gca_b200 import abi, mcts
    from oracle import oracle as orc
    from Algorithms.MCTS.config_single import Config as MctsConfig
    R, sims, depth, base = 65536, 100, 3, 11
    cfg = abi.make_mcts_config(MctsConfig)
    roots = _mcts_roots(R, seed=3)
    act, cn, cq, ca = mcts.search(roots, sims, depth, cfg=cfg, seed=2, root_id0=base, return_children=True)
    act, cn, cq, ca = act.cpu().numpy(), cn.cpu().numpy(), cq.cpu().numpy(), ca.cpu().numpy()
    host = roots.cpu().numpy()
    for r in _sample(R, 5):
        wb, wn, wq, wa = orc.mcts_search_philox(cfg, 80, host[r:r + 1], sims, depth, seed=2, root_id0=base + int(r))
        assert np.array_equal(ca[r], wa[0]) and np.array_equal(cn[r], wn[0]) and np.array_equal(cq[r], wq[0]), r
        assert np.array_equal(act[r], [wb[0] // 3, wb[0] % 3]), r


@pytest.mark.parametrize("R,random_intruders", [(4096, False), (2048, True)])
def test_mcts_playouts_bench_size_sampled_vs_oracle(R, random_intruders):
    """bench_mcts / bench_mctsrnd: 100 playouts of depth 3 per root on 4,096 roots (N = 80), and the random-intruder
    model on 2,048 roots taken from f32 observations."""
    from gca_b200 import abi, mcts
    from oracle import oracle as orc
    from Algorithms.MCTS.config_single import Config as MctsConfig
    P, depth, base = 100, 3, 1000
    cfg = abi.make_mcts_config(MctsConfig, random_intruders=random_intruders)
    roots = _mcts_roots(R, seed=2 if not random_intruders else 8, random_intruders=random_intruders)
    rw, first, fl = mcts.playouts(roots, P, depth=depth, cfg=cfg, seed=6, root_id0=base)
    rw, first, fl = rw.cpu().numpy(), first.cpu().numpy(), fl.cpu().numpy()
    host = roots.cpu().numpy()
    for r in _sample(R, 6):
        wr, wf, wfl = orc.mcts_playouts(cfg, 80, host[r:r + 1], P, depth, seed=6, root_id0=base + int(r))
        assert np.array_equal(fl[r], wfl[0]) and np.array_equal(first[r], wf[0]) and np.array_equal(rw[r], wr[0]), r
