"""MCTS forward model on the GPU: tape replay of the reference's recorded move() calls, and
bit-exact agreement of the Philox playout kernel with the CPU oracle."""
import os

import numpy as np
import pytest

from helpers import GOLDEN
from gca_b200 import abi

pytestmark = pytest.mark.gpu


def mcts_cfg(**over):
    from Algorithms.MCTS.config_single import Config
    c = abi.make_mcts_config(Config)
    for k, v in over.items():
        setattr(c, k, v)
    return c


RND = {"random_intruders": 1, "turn_prob": 0.1, "turn_max_deg": 10.0}     # the model of nodes_single_randintru.py


@pytest.mark.parametrize("stem,n", [("mcts", 3), ("mcts", 80), ("mctsrnd_model", 3), ("mctsrnd_model", 20)])
def test_move_replays_reference(stem, n):
    import torch
    from gca_b200 import mcts
    g = np.load(os.path.join(GOLDEN, "%s_n%d.npz" % (stem, n)))
    over = RND if stem != "mcts" else {}
    m = len(g["mv_root"])
    states = torch.as_tensor(g["roots"][g["mv_root"]].copy(), device="cuda")
    actions = torch.as_tensor((g["mv_action"][:, 0] * 3 + g["mv_action"][:, 1]).astype(np.int32), device="cuda")
    tape = torch.as_tensor(np.nan_to_num(g["mv_tape"], nan=0.0), device="cuda")
    cursor = torch.zeros(m, dtype=torch.int64, device="cuda")
    flags = mcts.move(states, actions, mcts_cfg(**over), tape=tape, cursor=cursor).cpu().numpy()
    assert np.array_equal(cursor.cpu().numpy(), g["mv_tape_len"])
    assert np.array_equal((flags & abi.MCTS_WALL) != 0, g["mv_hit_wall"])
    assert np.array_equal((flags & abi.MCTS_CONFLICT) != 0, g["mv_conflict"])
    assert np.array_equal((flags & abi.MCTS_GOAL) != 0, g["mv_reach_goal"])
    out = states.cpu().numpy()
    # heading noise comes from the tape; cos/sin are the only non-shared ops: <= 1e-9 relative, almost always exact
    assert np.allclose(out, g["mv_out_state"], rtol=1e-9, atol=1e-300)
    print("bit-identical successor states: %d / %d" % (int((out == g["mv_out_state"]).all(1).sum()), m))


@pytest.mark.parametrize("n,roots_n,playouts,depth,over", [
    (80, 64, 100, 3, {}), (3, 200, 50, 3, {}), (1, 50, 20, 2, {}), (0, 50, 20, 3, {}),
    (200, 16, 30, 3, {}),                                   # 200 intruders: 2 roots per CTA
    (80, 8, 10, 4, {"simulate_frame": 10}),                 # 40 sub-frames: two lane chunks
    (20, 32, 20, 3, {"speed_sigma": 0.05, "position_sigma": 0.3}),
    (80, 48, 40, 3, RND), (3, 100, 50, 3, RND), (1, 40, 20, 2, RND), (0, 20, 10, 3, RND),
    (33, 24, 20, 4, dict(RND, speed_sigma=0.05, position_sigma=0.3, turn_prob=0.5)),
    (80, 21, 100, 3, RND),                                  # 2 roots per CTA, ragged last CTA
    (5, 7, 30, 3, dict(RND, speed_sigma=0.05, position_sigma=0.3, turn_prob=0.5)),
])
def test_playouts_bit_exact_vs_oracle(n, roots_n, playouts, depth, over):
    import torch
    from gca_b200 import mcts
    from oracle import oracle as orc
    cfg = mcts_cfg(**over)
    rng = np.random.RandomState(n + 7)
    roots = _random_roots(n, roots_n, n + 7, six=bool(over.get("random_intruders")))
    fa = rng.randint(-1, 9, (roots_n, playouts)).astype(np.int8)
    want_r, want_f, want_fl = orc.mcts_playouts(cfg, n, roots, playouts, depth, first_action=fa, seed=77, root_id0=5)
    got_r, got_f, got_fl = mcts.playouts(torch.as_tensor(roots, device="cuda"), playouts, depth=depth, cfg=cfg,
                                         first_action=torch.as_tensor(fa, device="cuda"), seed=77, root_id0=5)
    assert np.array_equal(got_fl.cpu().numpy(), want_fl)
    assert np.array_equal(got_f.cpu().numpy(), want_f)
    assert np.array_equal(got_r.cpu().numpy(), want_r)
    print("n=%d flags histogram" % n, np.bincount(want_fl.ravel(), minlength=5).tolist())


NOISE = {"speed_sigma": 0.05, "position_sigma": 0.3}


@pytest.mark.parametrize("n,roots_n,playouts,depth,over", [
    (20, 16, 30, 3, NOISE), (50, 12, 30, 3, NOISE), (80, 12, 30, 3, NOISE), (120, 8, 20, 3, NOISE),
    (200, 6, 20, 3, NOISE),
    (100, 8, 40, 3, RND), (100, 6, 20, 3, dict(RND, **NOISE)), (80, 5, 300, 3, RND),
])
def test_warp_per_playout_kernel_bit_exact(n, roots_n, playouts, depth, over):
    """Position noise takes the warp-per-playout kernel: mcts_playout_kernel<1..4> for up to 32..128 intruders, <0>
    beyond.  So does the random-intruder model with more than 80 intruders or more than 256 playouts per root
    (mcts_playout_kernel<0, true>; culled without noise, as in the last case)."""
    test_playouts_bit_exact_vs_oracle(n, roots_n, playouts, depth, over)


@pytest.mark.parametrize("n,roots_n,playouts,depth", [
    (80, 37, 100, 3), (3, 9, 50, 3), (80, 5, 500, 2),
    (80, 5, 1100, 2), (3, 4, 1008, 3),
    (80, 9, 40, 0), (80, 3, 1100, 0),
])
def test_packed_kernel_bit_exact(n, roots_n, playouts, depth):
    """position_sigma == 0 takes mcts_playout_packed_kernel: several roots per CTA (37 roots of 100 playouts = a ragged
    last CTA), one root per CTA (500 playouts), one root in slices of 512 playouts (1100 = three slices, the last one
    ragged), and depth 0 (the reward of the root state itself)."""
    test_playouts_bit_exact_vs_oracle(n, roots_n, playouts, depth, {})


def _random_roots(n, roots_n, seed, six=False):
    """Raw observations: 4 values per intruder (Simulators/SingleAircraftMCTSEnv), or six - + speed, heading - for the
    random-intruder model."""
    rng = np.random.RandomState(seed)
    roots = _random_roots4(n, roots_n, rng)
    if not six:
        return roots
    out = np.zeros((roots_n, 6 * n + 8))
    out[:, 6 * n:] = roots[:, 4 * n:]
    it = roots[:, :4 * n].reshape(roots_n, n, 4)
    speed = np.hypot(it[..., 2], it[..., 3])
    heading = np.arctan2(it[..., 3], it[..., 2])
    out[:, :6 * n] = np.concatenate([it, speed[..., None], heading[..., None]], -1).reshape(roots_n, 6 * n)
    return out


def _random_roots4(n, roots_n, rng):
    L = 4 * n + 8
    roots = np.zeros((roots_n, L))
    for r in range(roots_n):
        ip = rng.uniform(0, 800, (n, 2)); sp = rng.uniform(5 / 3, 8 / 3, n); hd = rng.uniform(0, 2 * np.pi, n)
        roots[r, :4 * n] = np.stack([ip[:, 0], ip[:, 1], sp * np.cos(hd), sp * np.sin(hd)], -1).ravel()
        own = rng.uniform(30, 770, 2); h = rng.uniform(0, 2 * np.pi); s = rng.uniform(5 / 3, 8 / 3)
        goal = own + rng.uniform(-120, 120, 2) if r % 3 == 0 else rng.uniform(0, 800, 2)
        if n and r % 4 == 1:                                  # aim at an intruder: conflicts
            own = ip[rng.randint(max(n - 1, 1))] - 30 * np.array([np.cos(h), np.sin(h)])
        if r % 7 == 2:                                        # near a wall, heading out
            own = np.array([rng.uniform(0.5, 15), rng.uniform(100, 700)]); h = np.pi + rng.normal(0, .2)
        roots[r, 4 * n:] = [own[0], own[1], s * np.cos(h), s * np.sin(h), s, h, goal[0], goal[1]]
    return roots


@pytest.mark.parametrize("n,roots_n,sims,depth,over", [
    (80, 96, 100, 3, {}), (3, 64, 100, 3, {}), (1, 40, 30, 2, {}), (0, 40, 50, 3, {}), (200, 12, 40, 3, {}),
    (80, 16, 200, 4, {}), (20, 40, 60, 3, {"speed_sigma": 0.05}), (80, 8, 0, 3, {}), (80, 8, 5, 3, {}),
])
def test_device_tree_search_bit_exact_vs_oracle(n, roots_n, sims, depth, over):
    """gca_mcts_search (device-resident UCT trees, one lane per root) against the oracle's best_action() with the same
    Philox draws: the chosen action and the visit counts / value sums of every root child, bit for bit."""
    import torch
    from gca_b200 import mcts
    from oracle import oracle as orc
    cfg = mcts_cfg(**over)
    roots = _random_roots(n, roots_n, n + 11)
    want_b, want_n, want_q, want_a = orc.mcts_search_philox(cfg, n, roots, sims, depth, seed=123, root_id0=9)
    act, cn, cq, ca = mcts.search(torch.as_tensor(roots, device="cuda"), sims, depth, cfg=cfg, seed=123, root_id0=9,
                                  return_children=True)
    assert np.array_equal(ca.cpu().numpy(), want_a)
    assert np.array_equal(cn.cpu().numpy(), want_n)
    assert np.array_equal(cq.cpu().numpy(), want_q)
    best = want_b.astype(np.int64)
    assert np.array_equal(act.cpu().numpy(), np.stack([best // 3, best % 3], -1))
    print("n=%d best-action histogram" % n, np.bincount(np.maximum(want_b, 0), minlength=9).tolist())


def test_device_tree_search_rejects_position_noise():
    import torch
    from gca_b200 import mcts
    with pytest.raises(abi.GcaError):
        mcts.search(torch.zeros((2, 16), dtype=torch.float64, device="cuda"), 10, 3, cfg=mcts_cfg(position_sigma=0.5))
    with pytest.raises(abi.GcaError):      # the random-intruder model: every playout moves its own intruders
        mcts.search(torch.zeros((2, 20), dtype=torch.float64, device="cuda"), 10, 3, cfg=mcts_cfg(**RND))


def test_drop_in_random_intruder_classes():
    """Agent_RandInt.py:37-41 call sequence on the drop-in classes of nodes_single_randintru.py (host tree, device
    move / rollout)."""
    from Algorithms.MCTS.nodes_single_randintru import SingleAircraftNode, SingleAircraftState
    from Algorithms.MCTS.search_single import MCTS
    g = np.load(os.path.join(GOLDEN, "mctsrnd_model_n3.npz"))
    np.random.seed(0)
    state = SingleAircraftState(state=g["roots"][0])
    root = SingleAircraftNode(state=state)
    best = MCTS(root).best_action(30, 2)
    assert best.state.prev_action in [(a, b) for a in range(3) for b in range(3)]
    assert len(root.children) == 9 and root.n == 30.0 and all(type(c) is SingleAircraftNode for c in root.children)
    nxt = state.move((1, 1))
    assert type(nxt) is SingleAircraftState and nxt.depth == 1 and nxt.state.shape == (6 * 3 + 8,)
    assert 0.0 <= nxt.reward() <= 1.0 and nxt.dist_intruder() > 0


def test_batched_agent_experiment():
    """Algorithms/MCTS/Agent.py run_experiment, batched: episodes finish, statistics are well formed, and planning
    beats a fixed action (fewer conflicts than flying straight)."""
    from gca_b200 import mcts
    out = mcts.run_experiment(num_envs=64, no_episodes=24, no_simulations=40, search_depth=3, seed=4, max_steps=1500)
    assert out["episodes"] >= 24 and out["searches"] > 0
    assert 0.0 <= out["nmac_prob"] <= 1.0 and 0.0 <= out["goal_prob"] <= 1.0
    assert out["goal_prob"] > 0.5, out
    print(out)


def test_batched_random_intruder_agent_experiment():
    """Agent_RandInt.py batched: the random-intruder env planned with root-parallel playouts of its own model."""
    from gca_b200 import mcts
    out = mcts.run_experiment(num_envs=48, no_episodes=12, no_simulations=36, search_depth=3, seed=5, max_steps=1200,
                              random_intruders=True)
    assert out["episodes"] >= 12 and out["searches"] > 0
    assert 0.0 <= out["nmac_prob"] <= 1.0 and out["goal_prob"] > 0.4, out
    print(out)


def test_drop_in_search_classes():
    """Agent.py:37-41 call sequence on the drop-in classes."""
    from Algorithms.MCTS.nodes_single import SingleAircraftNode, SingleAircraftState
    from Algorithms.MCTS.search_single import MCTS
    g = np.load(os.path.join(GOLDEN, "mcts_n3.npz"))
    np.random.seed(0)
    state = SingleAircraftState(state=g["roots"][0])
    root = SingleAircraftNode(state=state)
    best = MCTS(root).best_action(30, 2, device=False)         # the reference's structure: tree in Python objects
    assert best.state.prev_action in [(a, b) for a in range(3) for b in range(3)]
    assert len(root.children) == 9 and root.n == 30.0
    root2 = SingleAircraftNode(state=SingleAircraftState(state=g["roots"][0]))
    best2 = MCTS(root2).best_action(30, 2)                     # default: the whole search on the device
    assert best2.state.prev_action in [(a, b) for a in range(3) for b in range(3)]
    assert best2.parent is root2 and best2.state.depth == 1 and root2.children == [best2]
    nxt = state.move((1, 1))
    assert nxt.depth == 1 and nxt.prev_action == (1, 1) and nxt.state.shape == state.state.shape
    assert 0.0 <= nxt.reward() <= 1.0


def test_batched_planner_prefers_safe_actions():
    import torch
    from gca_b200 import mcts
    n = 3
    root = np.zeros(4 * n + 8)
    root[:12] = [400, 360, 0, 0, 700, 700, 0, 0, 100, 100, 0, 0]        # a stationary intruder straight ahead (north)
    root[12:] = [400, 300, 0, 2.5, 2.5, np.pi / 2, 400, 700]            # ownship heading north towards it and the goal
    acts = mcts.plan_actions(torch.as_tensor(np.tile(root, (16, 1)), device="cuda"), n_simulations=450, seed=1)
    assert acts.shape == (16, 2)
    assert (acts[:, 0] != 1).float().mean() > 0.8                        # going straight collides: the planner turns
