"""Small-batch exercise of every kernel for compute-sanitizer (memcheck / racecheck / initcheck).
Usage on the GPU box: compute-sanitizer --tool memcheck python tools/sanitize.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "gym-guidance-collision-avoidance-single_b200")]
import torch  # noqa: E402
from gca_b200.batched import BatchedAircraftEnv  # noqa: E402
from gca_b200.stack import ImageBatch  # noqa: E402
from gym_guidance_collision_avoidance_single.envs.config import Config  # noqa: E402

QUICK = os.environ.get("GCA_SANITIZE_QUICK") == "1"        # (one env variant only: the MCTS kernels are the subject)
for variant, B, N, mode in [("SingleAircraft2Env", 1000, 80, "fast"), ("SingleAircraftEnv", 77, 33, "fast"),
                            ("SingleAircraftHEREnv", 300, 80, "fast"), ("SingleAircraftEnv", 130, 7, "faithful"),
                            ("SingleAircraftEnv", 64, 0, "fast"), ("SingleAircraftDiscreteHEREnv", 90, 200, "fast")][:1 if QUICK else None]:
    env = BatchedAircraftEnv(variant, B, Config, n_intruders=N, mode=mode, seed=3)
    env.reset()
    for t in range(60):
        if env.continuous:
            a = torch.rand((B, 2), device="cuda", dtype=env.real) * 2 - 1
        else:
            a = torch.randint(0, 3, (B,), device="cuda", dtype=torch.int32)
        o, r, d, i = env.step(a, auto_reset=(t % 2 == 0))
        if t % 7 == 0 and bool(d.any()):
            env.reset(mask=d)
    env.observe()
    st = env.get_state()
    env.set_state(st)
    torch.cuda.synchronize()
    env.close()
    print("ok", variant, B, N, mode, flush=True)
img = ImageBatch(16, Config, n_intruders=20, frame_stack=4, seed=1)
img.reset()
for t in range(5):
    img.step(torch.randint(0, 9, (16,), device="cuda", dtype=torch.int32))
torch.cuda.synchronize()
print("ok stack")
img.close()

# Discrete9HER: random start + nearest-n observation kernel
from Simulators.config import Config as SimConfig  # noqa: E402
for B, N, mode in ((200, 80, "fast"), (70, 5, "faithful")):
    env = BatchedAircraftEnv("SingleAircraftDiscrete9HEREnv", B, SimConfig, n_intruders=N, mode=mode, seed=5)
    env.reset()
    for t in range(40):
        o, r, d, i = env.step(torch.randint(0, 9, (B,), device="cuda", dtype=torch.int32), auto_reset=(t % 2 == 0))
        if t % 5 == 0 and bool(d.any()):
            env.reset(mask=d)
    env.observe()
    env.counters()
    torch.cuda.synchronize()
    env.close()
    print("ok d9her", B, N, mode, flush=True)

# random-intruder env: heading / speed plane, drift instantiation of the streaming pass, turn + six-entry observation pass
rnd_roots = None
for B, N, mode in ((200, 80, "fast"), (70, 5, "faithful"), (45, 7, "fast"), (33, 1, "faithful")):
    env = BatchedAircraftEnv("SingleAircraftMCTSRandIntruderEnv", B, SimConfig, n_intruders=N, mode=mode, seed=6)
    env.reset()
    for t in range(40):
        o, r, d, i = env.step(torch.randint(0, 9, (B,), device="cuda", dtype=torch.int32), auto_reset=(t % 2 == 0))
        if t % 5 == 0 and bool(d.any()):
            env.reset(mask=d)
    env.observe()
    env.set_state(env.get_state())
    if rnd_roots is None:
        rnd_roots = env.obs[:24].double().contiguous().clone()
    torch.cuda.synchronize()
    env.close()
    print("ok mctsrnd", B, N, mode, flush=True)

# MCTS: both playout kernels, the move kernel, the device-resident search
from gca_b200 import abi, mcts, replay  # noqa: E402
from Algorithms.MCTS.config_single import Config as MctsConfig  # noqa: E402
cfg = abi.make_mcts_config(MctsConfig)
env = BatchedAircraftEnv("SingleAircraftMCTSEnv", 48, SimConfig, n_intruders=80, mode="faithful", seed=2)
roots = env.reset().clone()
env.close()
mcts.playouts(roots, 37, depth=3, cfg=cfg, seed=1)                  # packed kernel: 8 roots per CTA
mcts.playouts(roots[:13], 100, depth=3, cfg=cfg, seed=1)            # 5 roots per CTA, ragged last CTA
mcts.playouts(roots[:3], 1100, depth=2, cfg=cfg, seed=1)            # slices of 512 playouts, ragged last slice
mcts.playouts(roots[:5], 40, depth=0, cfg=cfg, seed=1)              # depth 0
ncfg = abi.make_mcts_config(MctsConfig)
ncfg.position_sigma, ncfg.speed_sigma = 0.3, 0.05
mcts.playouts(roots, 11, depth=3, cfg=ncfg, seed=1)                 # position noise: warp-per-playout kernel
mcts.search(roots, 60, 3, cfg=cfg, seed=4)
mcts.move(roots.clone(), torch.randint(0, 9, (48,), device="cuda", dtype=torch.int32), cfg)
rcfg = abi.make_mcts_config(MctsConfig, random_intruders=True)      # the nodes_single_randintru.py model
mcts.playouts(rnd_roots, 9, depth=3, cfg=rcfg, seed=1)              # lane-per-playout kernel, 8 roots per CTA
mcts.playouts(rnd_roots[:7], 100, depth=3, cfg=rcfg, seed=1)        # 2 roots per CTA, ragged last CTA
mcts.playouts(rnd_roots[:3], 300, depth=3, cfg=rcfg, seed=1)        # more than 256 playouts: warp-per-playout kernel
mcts.move(rnd_roots.clone(), torch.randint(0, 9, (24,), device="cuda", dtype=torch.int32), rcfg)
torch.cuda.synchronize()
print("ok mcts", flush=True)

# HER replay sampler, odd row widths
for dt, dim_o in ((torch.float32, 326), (torch.float64, 27), (torch.float32, 24)):
    E, T = 9, 13
    eb = {"o": torch.rand((E, T + 1, dim_o), device="cuda", dtype=dt), "u": torch.rand((E, T, 2), device="cuda", dtype=dt),
          "g": torch.rand((E, T, 2), device="cuda", dtype=dt), "ag": torch.rand((E, T + 1, 2), device="cuda", dtype=dt)}
    replay.sample_her_transitions(eb, 501, 4, 0.1, abi.OBS_DHER, seed=3, call=1)
torch.cuda.synchronize()
print("ok her replay")
