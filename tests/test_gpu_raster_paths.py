"""The StackEnv rasteriser (csrc/gca_raster.cu) on the paths that small square batches never reach, every pixel against
the CPU restatement (OracleEnv.raster) of the GPU's own state or of an oracle stepped alongside:

* the persistent loop: raster_kernel runs min(B, SMs x per_sm) CTAs and each one walks envs blockIdx.x,
  blockIdx.x + gridDim.x, ...; a CTA's second and later envs reuse its shared-memory plane after the previous bulk
  store has read it, reset the per-env cell masks and sprite counter, and zero-fill VecFrameStack planes meanwhile;
* the bench shape (65,536 envs x 80 intruders, 4-frame ring), on a sample of rows;
* canvases other than 800 x 800: non-square cell grids, 1 CTA per SM, the 4-byte copy that replaces the bulk store
  when the plane size is not a multiple of 16, a plane near the shared-memory limit, and canvases that are rejected;
* frame layouts chosen through the C ABI (gaps between planes and envs, an unaligned frames pointer), and the
  rejection of pointers the kernel's 4-byte accesses cannot use."""
import ctypes as C
import os

import numpy as np
import pytest

from gca_b200 import abi, sprites, variants

pytestmark = pytest.mark.gpu

GCA_ERR_INVALID, GCA_ERR_STATE = -1, -4            # include/gca.h
CANARY = 0xA5
PLANE = 200 * 200                                  # output plane of the 800 x 800 canvas


def _cfg(W=800, H=800):
    from gym_guidance_collision_avoidance_single.envs.config import Config
    if (W, H) == (800, 800):
        return Config
    return type("Cfg%dx%d" % (W, H), (Config,), dict(window_width=W, window_height=H))


def _sprites():
    return sprites.load_sprites(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sprites"))


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _smem_bytes(ow, oh):
    """raster_smem_bytes (csrc/gca_raster.cu): textures, plane, cell masks, poses / boxes, per-warp lists, summed-area
    tables and footprint classes.  Tied to the library by the byte count gca_raster reports for a canvas it rejects."""
    cells = ((ow + 15) // 16) * ((oh + 15) // 16)
    return 3 * 32 * 32 * 16 + ((ow * oh + 15) & ~15) + 16 * cells + 24 * 128 + 8 * 12 * 40 + 4 * 12 * 96 + \
        2 * 3 * 34 * 34 + ((3 * 33 * 33 + 15) & ~15)


def _launch_shape(W, H, B):
    """(CTAs per SM, grid) that launch_raster picks."""
    per_sm = 2 if 2 * _smem_bytes(W // 4, H // 4) + 2048 <= 227 * 1024 else 1
    return per_sm, min(B, _sm_count() * per_sm)


def _bulk_ok(plane, env_stride, plane_stride, frames_ptr):
    """launch_raster's condition for the bulk store (otherwise the plane leaves through 4-byte stores)."""
    return plane % 16 == 0 and env_stride % 16 == 0 and plane_stride % 16 == 0 and frames_ptr % 16 == 0


def _raster_call(batch, sprites_ptr, frames_ptr, env_stride, plane_stride, n_planes, slot, clear_mask):
    import torch
    return batch.lib.gca_raster(batch._h, sprites_ptr, frames_ptr, env_stride, plane_stride, n_planes, slot,
                                clear_mask.data_ptr() if clear_mask is not None else None,
                                C.c_void_p(torch.cuda.current_stream().cuda_stream))


def _oracle_frames(cfg_cls, st, rows, sp):
    """The restatement's frames of rows `rows` of a GPU state (get_state)."""
    from oracle import oracle as orc
    rows = np.asarray(rows)
    ref = orc.OracleEnv(variants.make_config("SingleAircraftStackEnv", cfg_cls), len(rows), st["ipos"].shape[1],
                        draws=1, trig=orc.TRIG_SHARED)
    for k, v in st.items():
        ref.state[k][...] = v[rows]
    return ref.raster(sp)


def _crowd(st, rng, W, H):
    """Sprites overlapping each other (ordered path, more than 4 live sprites on a pixel, deferred queue), on the
    canvas border and outside it - in envs spread over the whole batch, so over every CTA iteration."""
    B, n = st["ipos"].shape[0], st["ipos"].shape[1]
    rows = np.arange(B) % 2 == 0
    st["own_pos"][rows] = rng.uniform(-10, [W + 10, H + 10], (int(rows.sum()), 2))
    if n:
        st["ipos"][:, : n // 2] = (st["own_pos"][:, None, :] + rng.uniform(-40, 40, (B, n // 2, 2))).astype(np.float32)
    st["goal"][:] = st["own_pos"] + rng.uniform(-30, 30, (B, 2))


# ------------------------------------------------------------------------------- persistent loop
def test_frame_stack_ring_at_later_cta_iterations():
    """The VecFrameStack ring at B = 1000: envs finish at a CTA's later iterations, where their older planes are
    zero-filled while the bulk store of the CTA's previous env may still be in flight."""
    from test_gpu_raster import check_frame_stack_ring
    B = 1000
    assert B > 2 * _sm_count()
    assert check_frame_stack_ring(B) > 0


@pytest.mark.parametrize("mode", ["fast", "faithful"])
def test_envs_of_one_tile_on_different_position_planes(mode):
    """Masked resets without auto-reset advance the tick (and so flip the position plane) of the reset envs only: envs
    of one 32-env tile then read their intruders from different planes (counters[env].z & 1)."""
    import torch
    from gca_b200.stack import ImageBatch
    B, N = 1000, 80
    later = 2 * _sm_count()
    assert B > later
    sp = _sprites()
    env = ImageBatch(B, _cfg(), n_intruders=N, mode=mode, seed=21, sprites=sp)
    env.reset()
    rng = np.random.RandomState(6)
    finished = np.zeros(B, bool)
    checks = 0
    for t in range(6):
        st = env.batch.get_state()
        plant = np.arange(B) % 7 == t
        st["goal"][plant] = st["own_pos"][plant]
        env.batch.set_state({"goal": st["goal"]})
        _, _, done, _ = env.step(torch.as_tensor(rng.randint(0, 9, B).astype(np.int32), device="cuda"), auto_reset=False)
        finished |= done.cpu().numpy().astype(bool)
        if t % 3 == 2:
            assert finished[later:].any()
            env.batch.reset(mask=finished)
            finished[:] = False
            env._raster(None)
            st = env.batch.get_state()
            parity = np.concatenate([st["tick"] & 1, np.full(-B % 32, 2, np.uint32)]).reshape(-1, 32)
            mixed = [i for i, p in enumerate(parity) if len(set(p[p < 2])) == 2]
            assert any(32 * i >= later for i in mixed), mixed
            got = env.frame().cpu().numpy()[..., 0]
            want = _oracle_frames(_cfg(), st, np.arange(B), sp)
            assert np.array_equal(got, want), np.argwhere(got != want)[:4].tolist()
            checks += 1
    assert checks == 2
    env.close()


def test_bench_shape_ring_sampled():
    """bench_stack's shape: 65,536 envs x 80 intruders, FAST, Philox, auto-reset, 4-frame ring.  Before each step the
    goal is put on the ownship of one residue class of rows, so envs finish in every CTA iteration.  Rows sampled: the
    first and last 2 x SMs (every CTA's first and last env for 1 or 2 CTAs per SM), 512 seeded random rows, and up to
    256 of the rows that finished at the step; every plane of the ring against VecFrameStack made of oracle frames."""
    import torch
    from gca_b200.stack import ImageBatch
    B, N, k = 65536, 80, 4
    sms = _sm_count()
    edge = 2 * sms
    sp = _sprites()
    env = ImageBatch(B, _cfg(), n_intruders=N, frame_stack=k, seed=3, sprites=sp)
    rng = np.random.RandomState(17)
    fixed = np.unique(np.concatenate([np.arange(edge), np.arange(B - edge, B), rng.randint(edge, B - edge, 512)]))
    fixed_d = torch.as_tensor(fixed, device="cuda")

    def ring_rows(idx):                                  # [len, k, H, W], oldest plane first; only these rows are read
        return env.ring[idx][:, env.plane_order()].cpu().numpy()

    env.reset()
    model = np.zeros((len(fixed), k, 200, 200), np.uint8)
    model[:, -1] = _oracle_frames(_cfg(), env.batch.get_state(), fixed, sp)
    assert np.array_equal(ring_rows(fixed_d), model)
    for t in range(3):
        st = env.batch.get_state()
        plant = np.arange(B) % 61 == t
        st["goal"][plant] = st["own_pos"][plant]
        env.batch.set_state({"goal": st["goal"]})
        _, _, done, _ = env.step(torch.as_tensor(rng.randint(0, 9, B).astype(np.int32), device="cuda"))
        d = done.cpu().numpy().astype(bool)
        assert d[plant & (np.arange(B) >= edge)].any()     # (an intruder in conflict outranks the goal)
        st = env.batch.get_state()
        model = np.roll(model, -1, axis=1)               # vec_frame_stack.py:17-24
        model[d[fixed]] = 0
        model[:, -1] = _oracle_frames(_cfg(), st, fixed, sp)
        got = ring_rows(fixed_d)
        assert np.array_equal(got, model), (t, fixed[np.nonzero((got != model).any(axis=(1, 2, 3)))[0][:4]].tolist())
        fin = np.nonzero(d)[0]
        fin = np.sort(rng.choice(fin, min(256, len(fin)), replace=False))
        assert (fin >= edge).any()
        got = ring_rows(torch.as_tensor(fin, device="cuda"))
        assert not got[:, :-1].any(), t                  # a finished env starts from an all-zero stack
        assert np.array_equal(got[:, -1], _oracle_frames(_cfg(), st, fin, sp)), t
    env.close()


# ------------------------------------------------------------------------------- other canvases
# (W, H, B, CTAs per SM, bulk store): 640x480 non-square cell grid; 1024x768 grid of 148; 800x804 plane of 40,200
# bytes -> the 4-byte copy; 1600x1504 230,888 of 232,448 bytes of shared memory; 64x64 smaller than one sprite's reach
CANVASES = [(640, 480, 700, 2, True), (1024, 768, 400, 1, True), (800, 804, 700, 2, False), (1600, 1504, 300, 1, True),
            (64, 64, 40, 2, True)]


@pytest.mark.parametrize("W,H,B,per_sm,bulk", CANVASES)
def test_canvases_equal_cpu_restatement(W, H, B, per_sm, bulk):
    import torch
    from gca_b200.stack import ImageBatch
    from oracle import oracle as orc
    N = 80
    got_per_sm, grid = _launch_shape(W, H, B)
    assert got_per_sm == per_sm
    if W > 64:
        assert B > grid and B % grid != 0                # several envs per CTA, a ragged last wave
    cls = _cfg(W, H)
    sp = _sprites()
    env = ImageBatch(B, cls, n_intruders=N, mode="fast", seed=31, sprites=sp)
    plane = env.H * env.W                                # ImageBatch's ring with k = 1: both strides are one plane
    assert _bulk_ok(plane, plane, plane, env.ring.data_ptr()) == bulk
    ref = orc.OracleEnv(variants.make_config("SingleAircraftStackEnv", cls), B, N, draws=1, trig=orc.TRIG_SHARED,
                        seed=31, f32_positions=True, auto_reset=True)
    env.reset()
    ref.reset()
    rng = np.random.RandomState(W + H)
    st = env.batch.get_state()
    _crowd(st, rng, W, H)
    env.batch.set_state(st)
    for key, v in st.items():
        ref.state[key][...] = v
    env._raster(None)
    got, want = env.frame().cpu().numpy()[..., 0], ref.raster(sp)
    assert got.shape == (B, H // 4, W // 4)
    assert np.array_equal(got, want), np.argwhere(got != want)[:4].tolist()
    for t in range(2):
        a = rng.randint(0, 9, B).astype(np.int32)
        frame, _, _, info = env.step(torch.as_tensor(a, device="cuda"))
        ref.step(a)
        assert np.array_equal(info.cpu().numpy(), ref.info), t
    got, want = frame.cpu().numpy()[..., 0], ref.raster(sp)
    assert np.array_equal(got, want), np.argwhere(got != want)[:4].tolist()
    if W == 64:                                          # most output pixels have more than 4 live sprites
        assert (want != 255).mean() > 0.5
    env.close()


@pytest.mark.parametrize("W,H", [(1600, 1600), (808, 800)])
def test_canvas_rejected_without_launch(W, H):
    """A canvas whose plane does not fit in shared memory, and a width that is not a multiple of 16: GCA_ERR_STATE, no
    kernel, and the handle steps on."""
    import torch
    from gca_b200.stack import ImageBatch
    B = 8
    env = ImageBatch(B, _cfg(W, H), n_intruders=3, seed=1, sprites=_sprites())
    env.batch.reset()
    env.ring.fill_(CANARY)
    plane = env.H * env.W
    rc = _raster_call(env.batch, env.sprites.data_ptr(), env.ring.data_ptr(), plane, plane, 1, 0, None)
    assert rc == GCA_ERR_STATE
    msg = env.batch.lib.gca_last_error().decode()
    if W % 16 == 0:
        need = _smem_bytes(W // 4, H // 4)
        assert need > 227 * 1024
        assert "%dx%d" % (W, H) in msg and str(need) in msg, msg
    torch.cuda.synchronize()
    assert bool((env.ring == CANARY).all())
    tick = env.batch.counters()[:, 2].clone()
    env.batch.step(torch.zeros(B, dtype=torch.int32, device="cuda"))
    env.batch.check()
    assert bool((env.batch.counters()[:, 2] > tick).all())
    env.close()


# ------------------------------------------------------------------------------- frame layouts through the C ABI
@pytest.fixture(scope="module")
def abi_scene():
    """B = 700 envs with 80 intruders in a crowded state, the sprites on the device, the oracle's frames."""
    import torch
    from gca_b200.batched import BatchedAircraftEnv
    B, N = 700, 80
    assert B > 2 * _sm_count()
    sp = _sprites()
    batch = BatchedAircraftEnv("SingleAircraftStackEnv", B, _cfg(), n_intruders=N, mode="fast", seed=41)
    batch.reset()
    st = batch.get_state()
    _crowd(st, np.random.RandomState(8), 800, 800)
    batch.set_state(st)
    want = _oracle_frames(_cfg(), batch.get_state(), np.arange(B), sp)
    yield batch, torch.as_tensor(sp, device="cuda"), want
    batch.close()


# (plane_stride, env_stride, offset of frames in the buffer)
LAYOUTS = {"bulk_with_gaps": (PLANE + 16, 3 * (PLANE + 16) + 48, 64),
           "copy_with_gaps": (PLANE + 4, 3 * (PLANE + 4) + 8, 64),
           "copy_unaligned_frames": (PLANE, 3 * PLANE, 4)}


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_abi_frame_layouts(abi_scene, layout):
    """n_planes = 3, slot = 1, a third of the rows cleared, in a buffer of canary bytes: the slot plane is the oracle's
    frame, the other planes of a cleared row are zero, and no other byte - gaps, other planes of uncleared rows, bytes
    before and after - is written."""
    import torch
    batch, sp, want = abi_scene
    B, n_planes, slot = batch.num_envs, 3, 1
    ps, es, off = LAYOUTS[layout]
    total = off + (B - 1) * es + (n_planes - 1) * ps + PLANE + 64
    buf = torch.full((total,), CANARY, dtype=torch.uint8, device="cuda")
    base = buf.data_ptr()
    assert base % 16 == 0
    assert _bulk_ok(PLANE, es, ps, base + off) == (layout == "bulk_with_gaps")
    clear = (np.arange(B) % 3 == 1).astype(np.uint8)
    clear_d = torch.as_tensor(clear, device="cuda")
    abi.check(_raster_call(batch, sp.data_ptr(), base + off, es, ps, n_planes, slot, clear_d))
    got = buf.cpu().numpy()
    expect = np.full(total, CANARY, np.uint8)
    for e in range(B):
        for pl in range(n_planes):
            at = off + e * es + pl * ps
            if pl == slot:
                expect[at: at + PLANE] = want[e].ravel()
            elif clear[e]:
                expect[at: at + PLANE] = 0
    bad = np.nonzero(got != expect)[0]
    assert len(bad) == 0, (len(bad), bad[:4].tolist(), [((b - off) // es, (b - off) % es) for b in bad[:4]])


@pytest.mark.parametrize("which", ["frames", "sprites"])
def test_unaligned_pointer_rejected(abi_scene, which):
    """The kernel reads sprites and writes frames in 4-byte words: a pointer that is not 4-byte aligned is GCA_ERR_INVALID,
    named in the message, and nothing is launched."""
    import torch
    batch, sp, _ = abi_scene
    B = batch.num_envs
    buf = torch.full((3 * B * PLANE + 64,), CANARY, dtype=torch.uint8, device="cuda")
    sp_buf = torch.zeros(sp.numel() + 16, dtype=torch.uint8, device="cuda")
    shift = 1 if which == "sprites" else 0
    sp_buf[shift: shift + sp.numel()] = sp.reshape(-1)
    frames = buf.data_ptr() + (2 if which == "frames" else 0)
    rc = _raster_call(batch, sp_buf.data_ptr() + shift, frames, 3 * PLANE, PLANE, 3, 1,
                      torch.ones(B, dtype=torch.uint8, device="cuda"))
    assert rc == GCA_ERR_INVALID
    msg = batch.lib.gca_last_error().decode()
    assert msg.startswith(which) and "aligned" in msg, msg
    torch.cuda.synchronize()
    assert bool((buf == CANARY).all())
