"""Adaptive sampling (rt_render_adaptive, ray_tracing_series_rust_b200/adaptive.py).

CPU: the numpy reference's error and dilation against hand-computed values and a brute force, the reference driven by the oracle's
sample-range renders (threshold 0 = the full render, a huge threshold stops every pixel at the first check point, sample maps are
monotone in the threshold and every pixel holds exactly the sums of its own samples), resolve_accumulator with per-pixel counts, and
the argument checks of the entry point on a scene that is not committed.
GPU: rt_render_adaptive at threshold 0 is rt_render bit for bit in every render mode; above 0 it equals the numpy reference over
rt_render sample ranges exactly (sums, sample counts, Screen), in every render mode."""
import ctypes as C
import os

import numpy as np
import pytest

import ray_tracing_series_rust_b200 as rtb
from ray_tracing_series_rust_b200 import adaptive, capi
from ray_tracing_series_rust_b200.animation import resolve_accumulator

RT_ERR_INVALID, RT_ERR_STATE = -1, -2
FLAGS = {"wavefront": 4, "fused": 8, "pool": 16, "auto": 0}


def check_points(spp, min_samples, step):
    return [n for n in range(2 * step, spp, 2 * step) if n >= min_samples]


def rounds_sum(render_range, n, step):
    """Sum of the round renders [0, step), [step, 2 step), ... up to n samples."""
    return sum(render_range(s0, min(s0 + step, n)) for s0 in range(0, n, step))


# ---------------------------------------------------------------- numpy reference


def test_half_buffer_error_hand_values():
    S = 4294967296.0
    A = np.array([[[3, 4, 5], [0, 0, 0]]], dtype=np.int64) * (1 << 32)
    B = np.array([[[1, 4, 9], [0, 0, 0]]], dtype=np.int64) * (1 << 32)
    err = adaptive.half_buffer_error(A, B, 2)
    # pixel 0: d = 2 + 0 + 4 = 6 (x 2^32), t = 4 + 8 + 14 = 26 (x 2^32), S = 2 * 2^32
    assert err[0, 0] == (6.0 / 2.0) / np.sqrt(1e-4 + 26.0 / 4.0)
    assert err[0, 1] == 0.0
    # the exact order of operations, on sums that are not multiples of 2^32
    a = np.array([[[123456789, 987654321, 5]]], dtype=np.int64)
    b = np.array([[[123456000, 987000000, 7]]], dtype=np.int64)
    h = 3
    d = (abs(123456789.0 - 123456000.0) + abs(987654321.0 - 987000000.0)) + abs(5.0 - 7.0)
    t = ((123456789.0 + 123456000.0) + (987654321.0 + 987000000.0)) + (5.0 + 7.0)
    want = (d / (h * S)) / np.sqrt(1e-4 + t / (2.0 * (h * S)))
    assert adaptive.half_buffer_error(a, b, h)[0, 0] == want


def _brute_next(active, err, tau, radius, rows):
    H, W = active.shape
    out = np.zeros_like(active)
    for y in range(H):
        for x in range(W):
            if not active[y, x]:
                continue
            for yy in range(max(0, y - radius), min(rows, y + radius + 1)):
                for xx in range(max(0, x - radius), min(W, x + radius + 1)):
                    if active[yy, xx] and not (err[yy, xx] < tau):
                        out[y, x] = True
    return out


@pytest.mark.parametrize("radius", [0, 1, 2, 3])
def test_next_active_matches_brute_force(radius):
    rng = np.random.default_rng(radius)
    for trial in range(6):
        H, W = int(rng.integers(5, 14)), int(rng.integers(5, 14))
        rows = H if trial % 2 == 0 else int(rng.integers(1, H))  # odd trials: unrendered compat_threads rows on top
        active = rng.random((H, W)) < 0.7
        active[rows:] = False
        err = rng.random((H, W))
        err[rng.random((H, W)) < 0.05] = np.nan  # NaN never counts as converged
        tau = 0.85
        got = adaptive.next_active(active, err, tau, radius, rows)
        assert np.array_equal(got, _brute_next(active, err, tau, radius, rows))
        assert not (got & ~active).any()


def test_resolve_accumulator_per_pixel_counts():
    rng = np.random.default_rng(1)
    acc = rng.integers(0, 40 << 32, size=(6, 5, 3), dtype=np.int64)
    uniform = resolve_accumulator(acc, 24)
    assert np.array_equal(resolve_accumulator(acc, np.full((6, 5), 24, np.int32)), uniform)
    counts = rng.integers(1, 30, size=(6, 5)).astype(np.int32)
    got = resolve_accumulator(acc, counts)
    for y in range(6):
        for x in range(5):
            assert np.array_equal(got[y, x], resolve_accumulator(acc[y:y + 1, x:x + 1], int(counts[y, x]))[0, 0])
    counts[0] = 0
    acc[0] = 0
    assert not resolve_accumulator(acc, counts)[0].any()  # 0 samples (an unrendered row): black


@pytest.fixture(scope="module")
def oracle_book1(orc):
    """Book-1 classic (scene 13), 48 x 32, 24 spp: the oracle's sample-range renders, cached.  The oracle rounds a pixel's sum to
    fixed point once per call (the library once per sample), so a sum of its range renders can differ from its one-call render by one
    unit (2^-32) per range: the reference is compared with sums of the same round renders, and with the one-call render within that."""
    W, aspect, spp = 48, 1.5, 24
    o = orc.new_scene()
    o.world_build(13, 0xB001)
    o.commit()
    H = o.image_height(capi.make_config(W, aspect, spp, 50))
    cache = {}

    def render_range(s0, s1):
        if (s0, s1) not in cache:
            cfg = capi.make_config(W, aspect, spp, 50, seed=3, sample_begin=s0, sample_end=s1)
            cache[(s0, s1)] = o.render(cfg, want_accum=True)[1]
        return cache[(s0, s1)]

    return render_range, (H, W, 3), spp


def test_reference_threshold_zero_is_the_full_render(oracle_book1):
    render_range, shape, spp = oracle_book1
    for radius in (0, 2):
        acc, smp = adaptive.adaptive_reference(render_range, shape, shape[0], spp, 8, 4, 0.0, radius)
        assert np.array_equal(acc, rounds_sum(render_range, spp, 4))
        assert np.abs(acc - render_range(0, spp)).max() <= spp // 4
        assert (smp == spp).all()


def test_reference_huge_threshold_stops_at_the_first_check_point(oracle_book1):
    render_range, shape, spp = oracle_book1
    for min_samples, first in ((0, 8), (8, 8), (9, 16), (16, 16)):
        acc, smp = adaptive.adaptive_reference(render_range, shape, shape[0], spp, min_samples, 4, 1e30, 1)
        assert (smp == first).all()
        assert np.array_equal(acc, rounds_sum(render_range, first, 4))


def test_reference_sample_maps_are_monotone_and_exact(oracle_book1):
    render_range, shape, spp = oracle_book1
    H = shape[0]
    for radius in (0, 1):
        prev = None
        for tau in (0.0, 0.1, 0.3, 0.5, 1e30):
            acc, smp = adaptive.adaptive_reference(render_range, shape, H, spp, 8, 4, tau, radius)
            assert set(np.unique(smp)) <= set(check_points(spp, 8, 4)) | {spp}
            if prev is not None:
                assert (smp <= prev).all()  # a larger threshold never renders a pixel longer
            prev = smp
            for n in np.unique(smp):  # every pixel holds exactly the sums of its own first samples
                m = smp == n
                assert np.array_equal(acc[m], rounds_sum(render_range, int(n), 4)[m])
            if tau == 0.3:
                assert len(np.unique(smp)) == 3, np.unique(smp, return_counts=True)  # 8, 16 and 24 samples all occur


def test_reference_compat_rows_and_partial_last_round(oracle_book1):
    render_range, shape, spp = oracle_book1
    rows = shape[0] - 5
    acc, smp = adaptive.adaptive_reference(render_range, shape, rows, spp, 0, 5, 0.3, 1)  # rounds [0,5) .. [20,24): 24 = 4*5 + 4
    assert (smp[rows:] == 0).all() and not acc[rows:].any()
    assert set(np.unique(smp[:rows])) <= {10, 20, 24}


# ---------------------------------------------------------------- C-ABI argument checks (no GPU)


@pytest.fixture(scope="module")
def api():
    if not os.path.exists(rtb.LIB_PATH):
        rtb.build()
    api = rtb.load()
    fn = api.lib.rt_render_adaptive
    fn.restype, fn.argtypes = capi.RENDER_ADAPTIVE_SIGNATURE
    return api


def _call(api, scene, cfg, ac):
    return api.lib.rt_render_adaptive(scene.h, C.byref(cfg), C.byref(ac) if ac is not None else None, None, None, None, None)


def test_render_adaptive_argument_checks(api):
    s = rtb.new_scene()  # never committed: every rejection below comes from the argument checks
    cfg = capi.make_config(32, 1.0, 16, 5)
    good = dict(min_samples=4, step=2, threshold=0.1, radius=1)

    def ac(**kw):
        d = dict(good)
        d.update(kw)
        return capi.AdaptiveConfig(d["min_samples"], d["step"], d["threshold"], d["radius"])

    bad = [None, ac(step=0), ac(step=-3), ac(threshold=-1e-9), ac(threshold=float("nan")), ac(threshold=float("inf")),
           ac(radius=-1), ac(radius=9), ac(min_samples=-1), ac(min_samples=17)]
    for a in bad:
        assert _call(api, s, cfg, a) == RT_ERR_INVALID
    for flags in ((1 << 16) | (2 << 24), 32):  # RT_RENDER_TILE_SHARD(1, 2), RT_RENDER_NO_WAIT
        assert _call(api, s, capi.make_config(32, 1.0, 16, 5, flags=flags), ac()) == RT_ERR_INVALID
    for s0, s1 in ((1, 0), (0, 8), (2, 16)):
        assert _call(api, s, capi.make_config(32, 1.0, 16, 5, sample_begin=s0, sample_end=s1), ac()) == RT_ERR_INVALID
    assert api.lib.rt_render_adaptive(None, C.byref(cfg), C.byref(ac()), None, None, None, None) == RT_ERR_INVALID
    assert api.lib.rt_render_adaptive(s.h, None, C.byref(ac()), None, None, None, None) == RT_ERR_INVALID
    # valid arguments (the bounds included, mode flags pass through): the scene state is what is wrong
    for a, c in ((ac(), cfg), (ac(min_samples=16, radius=8, threshold=0.0, step=1), cfg), (ac(min_samples=0), capi.make_config(32, 1.0, 16, 5, sample_end=16, flags=4 | 2)),
                 (ac(), capi.make_config(32, 1.0, 16, 5, flags=1 << 24))):  # RT_RENDER_TILE_SHARD(0, 1): one shard = no sharding, as in rt_render
        assert _call(api, s, c, a) == RT_ERR_STATE
    s.close()


def test_adaptive_config_layout():
    assert C.sizeof(capi.AdaptiveConfig) == 24
    assert capi.AdaptiveConfig.threshold.offset == 8 and capi.AdaptiveConfig.radius.offset == 16


# ---------------------------------------------------------------- GPU


def _gpu_scene(scene_id, param=0, seed=3):
    g = rtb.new_scene()
    g.world_build(scene_id, seed, param)
    g.commit()
    return g


def _range_renderer(g, W, aspect, spp, depth, seed, compat, flags=0):
    def render_range(s0, s1):
        cfg = capi.make_config(W, aspect, spp, depth, seed=seed, compat_threads=compat, sample_begin=s0, sample_end=s1, flags=flags)
        return g.render(cfg, want_accum=True)[1]
    return render_range


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,param,aspect", [(13, 0, 1.5), (99, 0, 16 / 9), (14, 48, 1.0), (5, 0, 1.0), (6, 0, 1.0)])
def test_threshold_zero_is_rt_render_bit_for_bit(scene_id, param, aspect):
    g = _gpu_scene(scene_id, param)
    W, spp = 72, 14
    for mode, flags in FLAGS.items():
        cfg = capi.make_config(W, aspect, spp, 50, seed=4, flags=flags)
        sr, ar, str_ = g.render(cfg, want_accum=True)
        sa, aa, smp, sta = g.render_adaptive(cfg, 0.0, min_samples=0, step=3, radius=1)
        assert np.array_equal(aa, ar), mode
        assert np.array_equal(sa, sr), mode
        assert (smp == spp).all(), mode
        assert sta["paths"] == str_["paths"] == smp.sum() and sta["segments"] == str_["segments"], mode
    g.close()


ADAPTIVE_CASES = [  # scene, aspect, W, spp, min_samples, step, threshold, radius, compat_threads
    (13, 1.5, 64, 24, 8, 4, 0.3, 0, 0),
    (13, 1.5, 64, 24, 8, 4, 0.3, 2, 0),
    (4, 1.0, 56, 24, 0, 4, 0.5, 0, 0),
    (4, 1.0, 56, 24, 0, 4, 0.5, 2, 0),
    (6, 1.0, 56, 20, 6, 3, 0.5, 0, 0),   # 20 spp in rounds of 3: the last round traces one sample
    (6, 1.0, 56, 20, 6, 3, 0.5, 2, 0),
    (13, 1.5, 64, 22, 0, 2, 0.2, 1, 5),  # compat_threads = 5: 42 = 8 * 5 + 2 rows, the top two black with 0 samples
]


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,aspect,W,spp,min_samples,step,tau,radius,compat", ADAPTIVE_CASES)
def test_adaptive_equals_numpy_reference(scene_id, aspect, W, spp, min_samples, step, tau, radius, compat):
    g = _gpu_scene(scene_id)
    cfg0 = capi.make_config(W, aspect, spp, 50, seed=6, compat_threads=compat)
    H = g.image_height(cfg0)
    rows = (H // compat) * compat if compat else H
    ref_acc, ref_smp = adaptive.adaptive_reference(_range_renderer(g, W, aspect, spp, 50, 6, compat), (H, W, 3), rows, spp, min_samples, step,
                                                   tau, radius)
    ref_screen = resolve_accumulator(ref_acc, ref_smp)
    assert len(np.unique(ref_smp[:rows])) >= 2, "the case must exercise convergence"
    if compat:
        assert rows < H and (ref_smp[rows:] == 0).all()
    for mode, flags in FLAGS.items():
        cfg = capi.make_config(W, aspect, spp, 50, seed=6, compat_threads=compat, flags=flags)
        screen, acc, smp, st = g.render_adaptive(cfg, tau, min_samples=min_samples, step=step, radius=radius)
        assert np.array_equal(smp, ref_smp), mode
        assert np.array_equal(acc, ref_acc), mode
        assert np.array_equal(screen, ref_screen), mode
        assert st["paths"] == int(smp.sum()), mode
    g.close()


@pytest.mark.gpu
def test_adaptive_buffers_are_reused_across_sizes():
    # the per-scene buffers grow for a larger image and are reused by a smaller one; results do not depend on the call history
    g = _gpu_scene(13)
    small = capi.make_config(40, 1.5, 12, 20, seed=2)
    first = g.render_adaptive(small, 0.3, min_samples=0, step=2, radius=1)
    g.render_adaptive(capi.make_config(120, 1.5, 6, 20, seed=2), 0.3, min_samples=0, step=2, radius=1)
    again = g.render_adaptive(small, 0.3, min_samples=0, step=2, radius=1)
    for a, b in zip(first[:3], again[:3]):
        assert np.array_equal(a, b)
    g.close()
