"""StackEnv image observation on the GPU: every pixel against the CPU restatement (the specification,
DESIGN.md 4.5), against frames of an independent renderer drawn with the reference's own sprites, the
4-frame ring against VecFrameStack's roll semantics, and the variant's reward / termination rules through the
facade."""
import numpy as np
import pytest

from gca_b200 import sprites, variants

pytestmark = pytest.mark.gpu


def _cfg():
    from gym_guidance_collision_avoidance_single.envs.config import Config
    return Config


def _sprite_set(which):
    import os
    if which == "reference":                                  # the reference's PNGs (committed as test vectors)
        return sprites.load_sprites(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sprites"))
    return sprites.default_sprites()


def test_frames_match_independent_renderer_gpu():
    """The CUDA rasteriser with the reference's sprites against frames that an independent renderer (float64 numpy +
    scipy bilinear, tests/golden/make_golden.py:render_independent) drew from states of the unmodified reference
    StackEnv, post-processed by the reference's own cv2 calls.  Bound stated in tests/test_raster_cpu.py."""
    from gca_b200.stack import ImageBatch
    from test_raster_cpu import check_frame, golden_frames
    g, sp = golden_frames()
    differ = 0
    for mode in ("fast", "faithful"):
        for k in range(len(g["n"])):
            n = int(g["n"][k])
            env = ImageBatch(3, _cfg(), n_intruders=n, mode=mode, seed=1, sprites=sp)
            env.reset()
            st = env.batch.get_state()
            st["own_pos"][:], st["own_hs"][:], st["goal"][:] = g["own_pos"][k], g["own_hs"][k], g["goal"][k]
            st["ipos"][:], st["ivel"][:] = g["ipos"][k][:n], g["ivel"][k][:n]
            st["ipos_is_f64"][:] = 0
            env.batch.set_state(st)
            env._raster(None)
            f = env.frame().cpu().numpy()[..., 0]
            for b in range(3):
                differ += check_frame(f[b], g["frame"][k], "%s frame %d (N = %d)" % (mode, k, n))
            env.close()
    print("pixels differing from the independent renderer:", differ)


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# B = 1000 (> 3 x 2 x 148, not a multiple of the persistent grid of either 1 or 2 CTAs per SM): every CTA rasterises
# several envs, so the crowded envs below land on a CTA's second and third iteration too
@pytest.mark.parametrize("n,B,mode,which", [(80, 24, "fast", "reference"), (80, 8, "faithful", "reference"), (0, 4, "fast", "reference"),
                                            (126, 6, "fast", "reference"), (5, 40, "fast", "reference"), (80, 24, "fast", "lookalike"),
                                            (33, 16, "faithful", "lookalike"), (80, 1000, "fast", "reference"),
                                            (80, 1000, "faithful", "lookalike"), (126, 1000, "fast", "reference"),
                                            (0, 1000, "fast", "reference")])
def test_frames_equal_cpu_restatement(n, B, mode, which):
    import torch
    from gca_b200.stack import ImageBatch
    from oracle import oracle as orc
    if B >= 1000:
        assert B >= 3 * 2 * _sm_count() and B % _sm_count() != 0
    sp = _sprite_set(which)
    env = ImageBatch(B, _cfg(), n_intruders=n, mode=mode, seed=11, sprites=sp)
    ref = orc.OracleEnv(variants.make_config("SingleAircraftStackEnv", _cfg()), B, n, draws=1, trig=orc.TRIG_SHARED,
                        seed=11, f32_positions=(mode == "fast"), auto_reset=True)
    f = env.reset().cpu().numpy()[..., 0]
    ref.reset()
    assert np.array_equal(f, ref.raster(sp))
    rng = np.random.RandomState(2)
    # crowd the scene: sprites overlapping each other, on the canvas border and outside it
    st = env.batch.get_state()
    st["own_pos"][: B // 2] = rng.uniform(-10, 810, (B // 2, 2))
    if n:
        st["ipos"][:, : n // 2] = st["own_pos"][:, None, :] + rng.uniform(-40, 40, (B, n // 2, 2))
        st["ipos"][:, : n // 2] = st["ipos"][:, : n // 2].astype(np.float32)
    st["goal"][:] = st["own_pos"] + rng.uniform(-30, 30, (B, 2))
    env.batch.set_state(st)
    for k, v in st.items():
        ref.state[k][...] = v
    for t in range(4):
        a = rng.randint(0, 9, B).astype(np.int32)
        fr, rew, done, info = env.step(torch.as_tensor(a, device="cuda"))
        ref.step(a)
        assert np.array_equal(info.cpu().numpy(), ref.info)
        assert np.array_equal(fr.cpu().numpy()[..., 0], ref.raster(sp)), t
    env.close()


def check_frame_stack_ring(B):
    """The k-plane ring against VecFrameStack's roll / zero-on-done semantics over 9 steps; returns how many envs past
    every CTA's first one (rows >= 2 x SMs) were zero-filled while all their older planes held a picture."""
    import torch
    from gca_b200.stack import ImageBatch
    k = 4
    cfg = _cfg()
    env = ImageBatch(B, cfg, n_intruders=20, frame_stack=k, seed=3, sprites=_sprite_set("reference"))
    first = env.reset().cpu().numpy()
    stacked = np.zeros((B, 200, 200, k), np.uint8)          # vec_frame_stack.py:26-30
    stacked[..., -1:] = first
    assert np.array_equal(env.stacked().cpu().numpy(), stacked)
    rng = np.random.RandomState(0)
    later = 2 * _sm_count()                                  # rows past every CTA's first env, for 1 or 2 CTAs per SM
    cleared_late = seen_done = 0
    for t in range(9):
        # the goal on the ownship: a residue class of rows, spread over the batch, finishes at this step -> stack reset
        # (unless an intruder inside the separation radius outranks the goal)
        st = env.batch.get_state()
        plant = np.arange(B) % 5 == t % 5
        st["goal"][plant] = st["own_pos"][plant]
        env.batch.set_state({"goal": st["goal"]})
        a = torch.as_tensor(rng.randint(0, 9, B).astype(np.int32), device="cuda")
        frame, rew, done, info = env.step(a)
        d = done.cpu().numpy().astype(bool)
        stacked = np.roll(stacked, shift=-1, axis=-1)        # vec_frame_stack.py:17-24
        # envs past every CTA's first one whose k - 1 older planes all hold a picture that the zero-fill must erase
        older = stacked[d & (np.arange(B) >= later)][..., :-1]
        cleared_late += int((older != 0).any(axis=(1, 2)).all(1).sum())
        stacked[d] = 0
        stacked[..., -1:] = frame.cpu().numpy()
        assert np.array_equal(env.stacked().cpu().numpy(), stacked), t
        assert d[plant].any(), t
        seen_done += int(d.sum())
    assert seen_done > 0
    env.close()
    return cleared_late


def test_frame_stack_ring_equals_vec_frame_stack():
    check_frame_stack_ring(12)


def test_stack_env_facade_rules():
    cfg = _cfg()
    cfg.intruder_size = 2
    cfg.max_steps = 5
    try:
        from gca_b200.stack import SingleAircraftStackEnv
        env = SingleAircraftStackEnv(seed=1, sprites=_sprite_set("reference"))
    finally:
        cfg.intruder_size = 0
        cfg.max_steps = 1000
    ob = env.reset()
    assert ob.shape == (200, 200, 1) and ob.dtype == np.uint8 and env.observation_space.shape == (200, 200, 1)
    assert (ob == 255).mean() > 0.95
    st = env.batch.get_state()
    st["own_pos"][0] = (799.5, 400.0)                        # about to leave the map, heading east
    st["own_hs"][0] = (0.0, 2.0)
    st["ipos"][0] = [[100, 100], [120, 700]]
    st["goal"][0] = (20.0, 20.0)
    env.batch.set_state(st)
    infos = []
    for _ in range(5):
        ob, r, done, info = env.step(4)
        infos.append((r, done, info))
    assert infos[0] == (-10, False, "w")                     # wall: -10 and NOT terminal (:170-171)
    assert infos[-1] == (0, True, "m") and env.steps == 5    # steps >= max_steps, checked first (:134-136)
    env.close()
