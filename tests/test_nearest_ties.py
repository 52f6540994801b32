"""The nearest-n observation of Simulators/SingleAircraftDiscrete{9,3}HEREnv.py with intruders at EXACTLY equal
distances: the order is (distance, index) - ties go to the lowest index - for every Config.n the ABI accepts, with f32
positions and with f32 / f64 positions mixed (a retried spawn keeps an f64 position; the two kinds compare by value).

The recorded traces hold no ties, so this pins the contract with a NumPy restatement of its own
(np.lexsort((index, distance))[:n]).  tie_states() is also the fixture of the device test of the same contract
(tests/test_gpu_config_paths.py): the kernel scans with four sub-lanes per env - 16-byte unit i // 2 in FAST mode,
i % 4 in FAITHFUL mode - and merges their lists, so the tied groups are spread over all four sub-lanes."""
import numpy as np
import pytest

from helpers import GOLDEN_VARIANTS, config_class
from gca_b200 import variants

# integer offsets with an integer length: the f32 subtraction, the squares and the square root are all exact
RINGS = {
    20: [(20, 0), (-20, 0), (0, 20), (0, -20), (12, 16), (16, -12), (-12, -16), (-16, 12), (12, -16), (-16, -12)],
    30: [(30, 0), (-30, 0), (0, 30), (0, -30), (18, 24), (24, -18), (-18, -24), (-24, 18), (18, -24), (-24, -18)],
    50: [(50, 0), (30, 40), (40, -30), (-30, -40), (0, -50), (-40, 30), (48, 14), (14, -48), (-48, -14), (-14, 48)],
}
TIE_VEL = (1.25, -0.5)      # few significant bits: exact in f32 and f64 adds, so duplicates stay tied after a step


def nearest_config(vk, n):
    """Config subclass with Config.n = n (the class attributes are snapshotted like the reference's Config idiom)."""
    base = config_class(vk)
    return type("CfgN%d" % n, (base,), {"n": n})


def tie_states(B, N, n, mixed, seed):
    """Canonical state dicts of B envs with N intruders: per env three rings of tied intruders at distances 20 / 30 / 50,
    the 30-ring straddling rank n (fewer than n intruders closer, at least n + 1 within it), at random - so out of
    distance order - indices; some ring members share a position (still tied after one step).  The other intruders sit
    60-140 px away at integer positions.  mixed: a random subset, ring members included, holds f64 positions."""
    from oracle import oracle as orc
    rng = np.random.RandomState(seed)
    st = orc.empty_state(B, N)
    st["own_vel_is_f32"][...] = 1
    for b in range(B):
        own = rng.randint(200, 600, 2).astype(np.float64)
        st["own_pos"][b] = own
        h = rng.uniform(0, 2 * np.pi)
        sp = rng.uniform(5 / 3, 8 / 3)
        st["own_hs"][b] = (h, sp)
        st["own_vel"][b] = (np.float32(sp * np.cos(h)), np.float32(sp * np.sin(h)))
        st["goal"][b] = rng.uniform(100, 700, 2)
        a = rng.randint(0, n)                                  # closer than the straddling ring
        t = rng.randint(n - a + 1, n - a + 5)                  # the ring at 30: a + t > n
        c = rng.randint(0, 4)
        idx = rng.permutation(N)[:a + t + c]
        offs = []
        for radius, count in ((20, a), (30, t), (50, c)):
            ring = RINGS[radius]
            pick = rng.randint(0, len(ring), count) if b % 2 else rng.permutation(len(ring))[:count] if count <= len(ring) \
                else rng.randint(0, len(ring), count)           # odd envs: duplicates on purpose
            offs += [ring[j] for j in pick]
        far = rng.uniform(60, 140, N) * np.exp(1j * rng.uniform(0, 2 * np.pi, N))
        pos = np.stack([np.round(own[0] + far.real), np.round(own[1] + far.imag)], -1)
        vel = rng.uniform(-2.5, 2.5, (N, 2)).astype(np.float32)
        for i, (dx, dy) in zip(idx, offs):
            pos[i] = (own[0] + dx, own[1] + dy)
            vel[i] = TIE_VEL
        st["ipos"][b] = pos
        st["ivel"][b] = vel
        if mixed:
            wide = rng.rand(N) < 0.4
            wide[idx[::2]] = True
            st["ipos_is_f64"][b] = wide
    st["ihs"][...] = 0.0
    return st


def restated_order(st, n):
    """np.lexsort((index, distance))[:n] per env, distances in the dtype the reference computes them in."""
    own = st["own_pos"].astype(np.float32)
    p = st["ipos"]
    dx32 = own[:, None, 0] - p[..., 0].astype(np.float32)
    dy32 = own[:, None, 1] - p[..., 1].astype(np.float32)
    d32 = np.sqrt(dx32 * dx32 + dy32 * dy32).astype(np.float64)
    dx64 = own[:, None, 0].astype(np.float64) - p[..., 0]
    dy64 = own[:, None, 1].astype(np.float64) - p[..., 1]
    d64 = np.sqrt(dx64 * dx64 + dy64 * dy64)                   # integer coordinates: exact, as the f64 norm
    d = np.where(st["ipos_is_f64"] != 0, d64, d32)
    N = p.shape[1]
    order = np.stack([np.lexsort((np.arange(N), row))[:n] for row in d])
    return order, d


def restated_rows(cfg, st, n):
    """The 5 n intruder entries of the observation from the restated order."""
    order, d = restated_order(st, n)
    B = order.shape[0]
    out = np.zeros((B, n, 5))
    W, H, diag = cfg.ob_window_width, cfg.ob_window_height, cfg.ob_diagonal
    ms = np.float32(cfg.max_speed)
    for b in range(B):
        for j, i in enumerate(order[b]):
            px, py = st["ipos"][b, i]
            if st["ipos_is_f64"][b, i]:
                out[b, j, 0], out[b, j, 1], out[b, j, 4] = px / W, py / H, d[b, i] / diag
            else:
                out[b, j, 0] = np.float32(px) / np.float32(W)
                out[b, j, 1] = np.float32(py) / np.float32(H)
                out[b, j, 4] = np.float32(d[b, i]) / np.float32(diag)
            v = st["ivel"][b, i]
            out[b, j, 2:4] = (v + ms) / np.float32(cfg.max_speed * 2)
    return out.reshape(B, 5 * n), order


def sublanes_of_ties(st, order, n, fast):
    """Distinct kernel sub-lanes that hold members of the tie group straddling rank n, per env."""
    _, d = restated_order(st, n + 1)
    out = []
    for b in range(order.shape[0]):
        members = np.nonzero(d[b] == d[b, order[b, n - 1]])[0]
        out.append(len(set(((members // 2) % 4 if fast else members % 4).tolist())))
    return np.array(out)


@pytest.mark.parametrize("vk", ["d9her", "d3her"])
@pytest.mark.parametrize("n", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("mixed", [False, True], ids=["f32", "mixed"])
def test_oracle_nearest_ties_lowest_index_first(vk, n, mixed):
    from oracle import oracle as orc
    B, N = 96, 40
    cfg = variants.make_config(GOLDEN_VARIANTS[vk], nearest_config(vk, n))
    assert cfg.nearest_n == n
    st = tie_states(B, N, n, mixed, seed=100 * n + mixed)
    ref = orc.OracleEnv(cfg, B, N, draws=1, trig=orc.TRIG_SHARED, f32_positions=not mixed)
    for k, v in st.items():
        ref.state[k][...] = v
    obs = ref.observe()
    want, order = restated_rows(cfg, st, n)
    assert np.array_equal(obs[:, 4:], want)
    # the fixture does what it is for: the tie at rank n is real and spread over the kernel's sub-lanes
    _, d = restated_order(st, n + 1)
    straddle = [d[b, order[b, n - 1]] == np.sort(d[b])[n] for b in range(B)]
    assert all(straddle)
    for fast in (True, False):
        lanes = sublanes_of_ties(st, order, n, fast)
        assert (lanes >= 2).mean() > 0.75 and lanes.max() == 4, (fast, np.bincount(lanes))
    if mixed:          # ties between an f32 and an f64 distance
        wide = st["ipos_is_f64"] != 0
        assert any(len(set(wide[b][d[b] == d[b, order[b, n - 1]]].tolist())) == 2 for b in range(B))
