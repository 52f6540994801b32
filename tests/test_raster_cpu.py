"""CPU checks of the image-observation specification: the cv2 half is pinned against the real
cv2 (the half of the reference that can run here); the GL half is pinned to an INDEPENDENT software
renderer (tests/golden/make_golden.py:render_independent - float64 numpy + scipy bilinear sampling, no code
or arithmetic shared with csrc/gca_raster_spec.h) on states taken from the unmodified reference StackEnv and
drawn with the reference's own sprite PNGs (DESIGN.md 4.5)."""
import os

import numpy as np
import pytest

from gca_b200 import sprites, variants
from oracle import oracle as orc


def _env(n=3):
    from gym_guidance_collision_avoidance_single.envs.config import Config
    cfg = variants.make_config("SingleAircraftStackEnv", Config)
    e = orc.OracleEnv(cfg, 1, n, draws=1, trig=orc.TRIG_SHARED, seed=4)
    e.reset()
    return e


def test_gray_and_area_resize_match_cv2():
    cv2 = pytest.importorskip("cv2")
    e = _env(6)
    e.state["own_pos"][0] = (400.3, 399.7)
    frames, rgb = e.raster(sprites.default_sprites(), want_rgb=True)
    want = cv2.resize(cv2.cvtColor(rgb[0], cv2.COLOR_RGB2GRAY), (200, 200), interpolation=cv2.INTER_AREA)
    assert np.array_equal(frames[0], want)                     # PKG/SingleAircraftStackEnv.py:104-108
    # and on arbitrary content (the sprites only exercise a few colours)
    rng = np.random.RandomState(0)
    img = rng.randint(0, 256, (800, 800, 3)).astype(np.uint8)
    wide = img.astype(np.int64)
    gray = ((9798 * wide[..., 0] + 19235 * wide[..., 1] + 3735 * wide[..., 2] + 16384) >> 15)
    assert np.array_equal(gray.astype(np.uint8), cv2.cvtColor(img, cv2.COLOR_RGB2GRAY))
    s = gray.reshape(200, 4, 200, 4).sum((1, 3))
    mine = (s + 7 + ((s >> 4) & 1)) >> 4
    assert np.array_equal(mine.astype(np.uint8), cv2.resize(gray.astype(np.uint8), (200, 200), interpolation=cv2.INTER_AREA))


def test_render_geometry():
    e = _env(1)
    sp = sprites.default_sprites()
    # park everything far apart: ownship heading north at (100, 700) -> top-left of the image
    e.state["own_pos"][0] = (100.0, 700.0)
    e.state["own_hs"][0] = (np.pi / 2, 2.0)
    e.state["goal"][0] = (600.0, 120.0)
    e.state["ipos"][0, 0] = (400.0, 400.0)
    e.state["ivel"][0, 0] = (2.0, 0.0)                           # heading east
    frames, rgb = e.raster(sp, want_rgb=True)
    f = frames[0]
    assert f.shape == (200, 200) and f.dtype == np.uint8
    assert (f == 255).mean() > 0.97                              # almost everything is background
    ys, xs = np.nonzero(f < 255)
    # three blobs around (x/4, (800-y)/4): ownship (25, 25), goal (150, 170), intruder (100, 100)
    for cx, cy in ((25, 25), (150, 170), (100, 100)):
        near = (np.abs(xs - cx) <= 5) & (np.abs(ys - cy) <= 5)
        assert near.sum() > 10
    assert np.all((np.abs(xs - 25) <= 5) & (np.abs(ys - 25) <= 5) | (np.abs(xs - 150) <= 5) & (np.abs(ys - 170) <= 5)
                  | (np.abs(xs - 100) <= 5) & (np.abs(ys - 100) <= 5))
    # heading north = rotation 0: the ownship quad reproduces the sprite unrotated (texel centres on pixel centres)
    quad = rgb[0, 100 - 16:100 + 16, 100 - 16:100 + 16].astype(np.float64)
    a = sp[0, :, :, 3:4].astype(np.float64) / 255
    expect = np.rint(sp[0, :, :, :3] * a + 255 * (1 - a))
    assert np.abs(quad - expect).max() <= 1
    # heading east = the sprite turned by -90 degrees: nose (top of the image) points right
    iq = rgb[0, 400 - 16:400 + 16, 400 - 16:400 + 16]
    assert np.abs(iq.astype(int) - np.rot90(np.rint(sp[2, :, :, :3] * (sp[2, :, :, 3:4] / 255.0) + 255 * (1 - sp[2, :, :, 3:4] / 255.0)), -1)).max() <= 1


@pytest.mark.parametrize("W,H,W2,H2", [(800, 800, 800, 804), (800, 800, 816, 800), (800, 800, 1600, 1504),
                                       (64, 64, 640, 480)])
def test_render_geometry_carries_to_other_canvases(W, H, W2, H2):
    """Only the 800 x 800 canvas is pinned against cv2 and the independent renderer.  A scene drawn on a W2 x H2 canvas
    with every y raised by H2 - H and x unchanged must give, in its first H/4 rows and W/4 columns, the frame of the
    W x H canvas: the top edge, the left edge and every sample stay where they were.  Positions are multiples of 1/256,
    so y + (H2 - H) and every sample's offset from a centre are exact in f32."""
    from gym_guidance_collision_avoidance_single.envs.config import Config
    B, N = 6, 40
    rng = np.random.RandomState(W2 * 7 + H2)
    q = lambda x: np.round(np.asarray(x) * 256.0) / 256.0
    envs = []
    for w, h in ((W, H), (W2, H2)):
        cls = type("Cfg%dx%d" % (w, h), (Config,), dict(window_width=w, window_height=h))
        envs.append(orc.OracleEnv(variants.make_config("SingleAircraftStackEnv", cls), B, N, draws=1,
                                  trig=orc.TRIG_SHARED, seed=4))
    st = envs[0].state
    # crowded, and across all four edges of the smaller canvas
    st["own_pos"][:] = q(rng.uniform(-20, [W + 20, H + 20], (B, 2)))
    st["own_hs"][:, 0] = rng.uniform(0, 2 * np.pi, B)
    st["goal"][:] = q(st["own_pos"] + rng.uniform(-30, 30, (B, 2)))
    st["ipos"][:, : N // 2] = q(st["own_pos"][:, None, :] + rng.uniform(-40, 40, (B, N // 2, 2)))
    st["ipos"][:, N // 2:] = q(rng.uniform(-20, [W + 20, H + 20], (B, N - N // 2, 2)))
    st["ivel"][:] = rng.uniform(-2, 2, (B, N, 2))
    lifted = envs[1].state
    for k, v in st.items():
        lifted[k][...] = v
    for k in ("own_pos", "goal", "ipos"):
        lifted[k][..., 1] += H2 - H
    assert np.array_equal(lifted["own_pos"][:, 1].astype(np.float64) - (H2 - H), st["own_pos"][:, 1])
    small, big = envs[0].raster(sprites.default_sprites()), envs[1].raster(sprites.default_sprites())
    assert big.shape == (B, H2 // 4, W2 // 4)
    assert np.array_equal(big[:, : H // 4, : W // 4], small)
    assert (small != 255).sum() > 1000                          # there is a picture to compare


def test_draw_order_later_sprites_on_top():
    e = _env(1)
    sp = sprites.default_sprites()
    e.state["own_pos"][0] = (400.0, 400.0)
    e.state["own_hs"][0] = (np.pi / 2, 2.0)
    e.state["goal"][0] = (100.0, 100.0)
    e.state["ipos"][0, 0] = (400.0, 400.0)                       # intruder exactly over the ownship
    e.state["ivel"][0, 0] = (0.0, 2.0)
    _, rgb = e.raster(sp, want_rgb=True)
    centre = rgb[0, 400, 400]
    assert centre[0] > 150 and centre[1] < 80                    # red intruder drawn after the yellow ownship


# stated bound of the picture against the independent renderer: <= 1 gray level on any pixel and >= 99.9 % of the
# pixels identical (measured: all 10 frames identical, 0 of 400,000 pixels differ)
FRAME_MAX_DIFF, FRAME_MIN_EQUAL = 1, 0.999


def golden_frames():
    here = os.path.dirname(os.path.abspath(__file__))
    g = np.load(os.path.join(here, "golden", "stack_frames.npz"))
    return g, sprites.load_sprites(os.path.join(here, "golden", "sprites"))


def check_frame(got, want, what=""):
    d = np.abs(got.astype(np.int32) - want.astype(np.int32))
    assert d.max() <= FRAME_MAX_DIFF and (d == 0).mean() >= FRAME_MIN_EQUAL, (what, int(d.max()), float((d == 0).mean()))
    return int((d != 0).sum())


def test_frames_match_independent_renderer():
    """The restatement (= the specification the CUDA rasteriser is pixel-exact to) against frames of reference states
    drawn by the independent renderer with the reference's PNGs, then the reference's own cv2 preprocess_frame."""
    from gym_guidance_collision_avoidance_single.envs.config import Config
    g, sp = golden_frames()
    cfg = variants.make_config("SingleAircraftStackEnv", Config)
    differ = 0
    for k in range(len(g["n"])):
        n = int(g["n"][k])
        e = orc.OracleEnv(cfg, 1, n, draws=1, trig=orc.TRIG_SHARED, seed=0)
        e.reset()
        e.state["own_pos"][0], e.state["own_hs"][0], e.state["goal"][0] = g["own_pos"][k], g["own_hs"][k], g["goal"][k]
        e.state["ipos"][0], e.state["ivel"][0] = g["ipos"][k][:n], g["ivel"][k][:n]
        differ += check_frame(e.raster(sp)[0], g["frame"][k], "frame %d (N = %d)" % (k, n))
        assert (g["frame"][k] != 255).sum() > 50                    # there is a picture to compare
    print("pixels differing from the independent renderer:", differ)
