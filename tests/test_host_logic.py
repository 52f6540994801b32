"""CPU-only checks: the C-ABI library loads and exports every symbol include/gca.h declares,
the host-side mirror of the reference interface (config table, spaces, registry, VecEnv state
machine) behaves like the reference, and the product refuses to run without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

from gca_b200 import abi, variants

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "gca.h")).read()
    declared = set(re.findall(r"^(?:int|const char\*)\s+(gca_[a-z0-9_]+)\s*\(", hdr, re.M))
    assert len(declared) >= 17
    lib = ctypes.CDLL(abi.LIB_PATH)
    missing = [name for name in sorted(declared) if not hasattr(lib, name)]
    assert not missing, missing
    assert abi.load().gca_abi_version() == abi.GCA_ABI_VERSION


def test_struct_layouts_match_header():
    assert ctypes.sizeof(abi.GcaConfig) == 21 * 8 + 8 * 4 + 8 + 16 + 8 + 3 * 8
    assert ctypes.sizeof(abi.GcaMctsConfig) == 10 * 8 + 4 * 4 + 2 * 8
    assert ctypes.sizeof(abi.GcaHostState) == 13 * 8 and ctypes.sizeof(abi.GcaOut) == 7 * 8
    assert ctypes.sizeof(abi.GcaTape) == 24


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from gca_b200.batched import BatchedAircraftEnv
    from gym_guidance_collision_avoidance_single.envs.config import Config
    with pytest.raises(abi.GcaError):
        BatchedAircraftEnv("SingleAircraftEnv", 4, Config)
    # the C ABI itself also refuses: no device -> GCA_ERR_CUDA, never a silent host path
    lib = abi.load()
    h = ctypes.c_void_p()
    cfg = variants.make_config("SingleAircraftEnv", Config)
    rc = lib.gca_create(ctypes.byref(cfg), 4, 0, abi.MODE_FAST, abi.DRAWS_PHILOX, 0, 0, 0, ctypes.byref(h))
    assert rc == -2 and b"CUDA" in lib.gca_last_error()
    import gym_guidance_collision_avoidance_single.envs as envs
    with pytest.raises(abi.GcaError):
        envs.SingleAircraftEnv()


def test_abi_argument_checking():
    lib = abi.load()
    from gym_guidance_collision_avoidance_single.envs.config import Config
    cfg = variants.make_config("SingleAircraftEnv", Config)
    h = ctypes.c_void_p()
    assert lib.gca_create(None, 4, 0, 1, 1, 0, 0, 0, ctypes.byref(h)) == -1
    assert lib.gca_create(ctypes.byref(cfg), 0, 0, 1, 1, 0, 0, 0, ctypes.byref(h)) == -1
    assert lib.gca_create(ctypes.byref(cfg), 4, -1, 1, 1, 0, 0, 0, ctypes.byref(h)) == -1
    assert lib.gca_create(ctypes.byref(cfg), 4, 0, 7, 1, 0, 0, 0, ctypes.byref(h)) == -1
    bad = variants.make_config("SingleAircraftEnv", Config)
    bad.obs_kind = 99
    assert lib.gca_create(ctypes.byref(bad), 4, 0, 1, 1, 0, 0, 0, ctypes.byref(h)) == -1
    assert b"obs_kind" in lib.gca_last_error()
    assert lib.gca_obs_dim(ctypes.byref(cfg), 80) == 328
    assert lib.gca_step(None, None, None, 1, None, None) == -1
    assert lib.gca_destroy(None) == 0


def test_variant_table_matches_reference_reward_rows():
    from gym_guidance_collision_avoidance_single.envs.config import Config
    from Simulators.config import Config as Sim
    rows = {k: variants.make_config(k, Sim if k not in ("SingleAircraftEnv", "SingleAircraft2Env", "SingleAircraftHEREnv", "SingleAircraftDiscreteHEREnv",
                                                     "SingleAircraftStackEnv") else Config)
            for k in variants.VARIANTS}
    r = rows["SingleAircraftDiscrete9HEREnv"]
    assert (r.obs_kind, r.random_start, r.nearest_n, r.ob_diagonal, r.wall_kind) == (abi.OBS_NEAREST, 1, 4, 800, abi.WALL_NONE)
    assert variants.obs_dim(r, 80) == 24
    r = rows["SingleAircraftEnv"]
    assert (r.r_nmac, r.r_conflict, r.r_goal, r.shaped_default, r.wall_kind) == (-20, -5, 10, 1, abi.WALL_NONE)
    r = rows["SingleAircraft2Env"]
    assert (r.r_nmac, r.r_conflict, r.r_wall, r.r_goal, r.wall_kind) == (-5, -1, -100, 1, abi.WALL_TERMINAL)
    r = rows["SingleAircraftHEREnv"]
    assert (r.r_nmac, r.r_conflict, r.r_goal, r.r_default, r.shaped_default) == (-5, -1, 0, -1, 0)
    r = rows["SingleAircraftDiscreteHEREnv"]
    assert (r.r_wall, r.r_goal, r.r_default, r.action_kind) == (-5, 1, 0, abi.ACT_DISCRETE3)
    r = rows["SingleAircraftStackEnv"]
    assert (r.r_wall, r.r_goal, r.wall_kind, r.max_steps, r.obs_kind) == (-10, 10000, abi.WALL_PENALTY, 1000, abi.OBS_NONE)
    r = rows["SingleAircraftMCTSEnv"]
    assert (r.r_nmac, r.r_conflict, r.r_goal, r.obs_kind, r.heading_sigma) == (-1.0, -0.5, 1.0, abi.OBS_RAW, np.radians(4))
    r = rows["SingleAircraftMCTSRandIntruderEnv"]      # Simulators/SingleAircraftMCTSRandIntruderEnv.py:133-140, :166-174, :183
    assert (r.obs_kind, r.intruder_turns, r.turn_prob, r.turn_max_deg, r.position_drift) == (abi.OBS_RAW6, 1, 0.1, 10.0, 10 / 30)
    assert variants.obs_dim(r, 80) == 488 and abi.load().gca_obs_dim(ctypes.byref(r), 80) == 488
    assert all(rows[k].intruder_turns == 0 and rows[k].position_drift == 0.0 for k in rows if k != "SingleAircraftMCTSRandIntruderEnv")
    from Algorithms.MCTS.config_single import Config as MctsConfig
    m = abi.make_mcts_config(MctsConfig, random_intruders=True)     # nodes_single_randintru.py:47, :64-65
    assert (m.random_intruders, m.turn_prob, m.turn_max_deg) == (1, 0.1, 10.0) and abi.make_mcts_config(MctsConfig).random_intruders == 0
    import Simulators.SingleAircraftMCTSRandIntruderEnv as rnd_mod
    import Algorithms.MCTS.nodes_single_randintru as rnd_nodes
    assert rnd_mod.SingleAircraftEnv.VARIANT == "SingleAircraftMCTSRandIntruderEnv"
    assert rnd_nodes.SingleAircraftState.RANDOM_INTRUDERS and rnd_nodes.SingleAircraftState.model_config().random_intruders == 1
    assert Config.intruder_size == 0 and Sim.intruder_size == 80          # Q28
    assert (Config.minimum_separation, Config.NMAC_dist, Config.initial_min_dist, Config.goal_radius) == (18.5, 5.0, 100.0, 20.0)
    assert variants.obs_dim(rows["SingleAircraftEnv"], 80) == 328 and variants.obs_dim(rows["SingleAircraftHEREnv"], 80) == 326


def test_every_variant_builds_its_config_from_its_default_config_class():
    """AircraftVecEnv(env, ..., config=None): the Config class comes from the variant table (the Simulators/ copies read
    Simulators/config.py: NMAC_penalty / sparse_reward / n / diagonal; the registered classes the package's)."""
    from gym_guidance_collision_avoidance_single.envs.config import Config
    from Simulators.config import Config as Sim
    for name in variants.VARIANTS:
        cls = variants.default_config_class(name)
        assert cls is (Config if name in ("SingleAircraftEnv", "SingleAircraft2Env", "SingleAircraftHEREnv",
                                          "SingleAircraftDiscreteHEREnv", "SingleAircraftStackEnv") else Sim), name
        c = variants.make_config(name, cls)                       # (raised AttributeError for four Simulators variants)
        assert abi.load().gca_obs_dim(ctypes.byref(c), 10) == variants.obs_dim(c, 10)
    assert variants.make_config("SingleAircraftDiscrete3HEREnv", Sim).action_kind == abi.ACT_DISCRETE3_HEADING


def test_sprite_resolution(tmp_path, monkeypatch):
    """gca_b200/sprites.py: the reference's PNGs when a checkout is known (argument or environment), else look-alikes
    with a warning."""
    from gca_b200 import sprites
    fix = os.path.join(ROOT, "tests", "golden", "sprites")
    monkeypatch.delenv("GCA_SPRITE_DIR", raising=False)
    monkeypatch.delenv("GCA_REFERENCE", raising=False)
    with pytest.warns(RuntimeWarning, match="look-alikes"):
        sp = sprites.resolve_sprites()
    assert np.array_equal(sp, sprites.default_sprites())
    real = sprites.resolve_sprites(sprite_dir=fix)
    assert real.shape == (3, 32, 32, 4) and not np.array_equal(real, sp)
    assert 0.35 < (real[0, :, :, 3] > 0).mean() < 0.5              # SURVEY appendix D: aircraft.png 40.5 % opaque
    monkeypatch.setenv("GCA_SPRITE_DIR", fix)
    assert np.array_equal(sprites.resolve_sprites(), real)
    monkeypatch.delenv("GCA_SPRITE_DIR")
    co = tmp_path / "checkout" / "gym_guidance_collision_avoidance_single" / "envs" / "images"
    co.mkdir(parents=True)
    for f in os.listdir(fix):
        (co / f).write_bytes(open(os.path.join(fix, f), "rb").read())
    monkeypatch.setenv("GCA_REFERENCE", str(tmp_path / "checkout"))
    assert np.array_equal(sprites.resolve_sprites(), real)
    with pytest.raises(FileNotFoundError):
        sprites.resolve_sprites(sprite_dir=str(tmp_path))
    assert np.array_equal(sprites.resolve_sprites(sprites=sp), sp)


def test_registry_and_spaces():
    import gym_guidance_collision_avoidance_single as pkg
    assert len(pkg.registry) == 5
    for spec in pkg.registry.values():
        assert spec["timestep_limit"] == 10000 and spec["reward_threshold"] == 10.0
    from gca_b200.spaces import Box, Discrete
    b = Box(low=-1, high=1, shape=(2,), dtype=float)
    assert b.contains(np.array([1.0, -1.0])) and not b.contains(np.array([1.0001, 0])) and not b.contains(np.zeros(3))
    pr = Box(low=np.array([0, 0]), high=np.array([800, 800]), dtype=np.float32)
    assert pr.contains(np.array([800.0, 0.0], np.float32)) and not pr.contains(np.array([800.0001, 5.0]))   # inclusive (Q6)
    assert Discrete(9).contains(8) and not Discrete(9).contains(9)


def test_oracle_struct_mirrors_and_bench_workload_config():
    """oracle/structs.py (the oracle's own mirror of include/gca.h, so that bench.py's reference arm needs nothing of
    the product) against the product's mirror, and its written-out workload config against the variant table."""
    from oracle import structs
    from gym_guidance_collision_avoidance_single.envs.config import Config
    for name in ("GcaConfig", "GcaHostState", "GcaMctsConfig"):
        a, b = getattr(abi, name), getattr(structs, name)
        assert ctypes.sizeof(a) == ctypes.sizeof(b)
        assert [(n, getattr(a, n).offset, getattr(a, n).size) for n, _ in a._fields_] == \
               [(n, getattr(b, n).offset, getattr(b, n).size) for n, _ in b._fields_], name
    import bench
    want = variants.make_config(bench.VARIANT, Config)
    got = structs.bench_workload_config()
    assert bytes(got) == bytes(want)
    src = open(os.path.join(ROOT, "oracle", "oracle.py")).read() + open(os.path.join(ROOT, "oracle", "structs.py")).read()
    assert "import gca_b200" not in src and "from gca_b200" not in src


def test_bench_reference_arm_runs_without_the_product():
    """`bench.py --impl reference`: oracle library only - neither libgca.so nor the gca_b200 package is loaded."""
    import json
    import subprocess
    import sys
    code = ("import sys, json; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '2', '--warmup', '1']; "
            "import bench; bench.run_cpu.__defaults__ = (64, 0.5); bench.main(); "
            "assert 'gca_b200' not in sys.modules and 'torch' not in sys.modules; "
            "maps = open('/proc/self/maps').read(); assert 'libgca.so' not in maps and 'libgca_oracle.so' in maps")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    assert set(line["config"]) == set(bench_config_keys())


def bench_config_keys():
    import bench
    return bench.workload_config().keys()


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: step()'s outputs as float .npy files under 64 MB, obs rows a fixed seeded sample."""
    import types
    import torch
    import bench
    B = bench.ENVS_PER_GPU
    g = torch.Generator().manual_seed(0)
    env = types.SimpleNamespace(num_envs=B, obs=torch.rand((B, 4 * bench.N_INTRUDERS + 8), generator=g),
                                reward=torch.rand((B,), generator=g),
                                done=torch.randint(0, 2, (B,), dtype=torch.uint8, generator=g),
                                info=torch.randint(0, 6, (B,), dtype=torch.uint8, generator=g))
    bench.dump_outputs(str(tmp_path / "a"), env)
    bench.dump_outputs(str(tmp_path / "b"), env)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["done.npy", "info.npy", "obs.npy", "obs_rows.npy", "reward.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    d = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    rows = d["obs_rows"].astype(np.int64)
    assert np.array_equal(d["obs"], env.obs.numpy()[rows]) and len(np.unique(rows)) == len(rows)
    for k in ("reward", "done", "info"):
        assert np.array_equal(d[k], getattr(env, k).numpy().astype(np.float32))
    assert all(np.array_equal(d[n[:-4]], np.load(tmp_path / "b" / n)) for n in names)


def test_bench_algorithmic_bytes():
    import bench
    assert bench.algorithmic_bytes_per_env_step(80) == 40 * 80 + 12 + 159
    assert bench.algorithmic_bytes_per_env_step(0, continuous=False) == 155
    assert bench.streaming_bytes_per_env_step(80) == 3200 and bench.handover_bytes_per_env_step(80) == 160
