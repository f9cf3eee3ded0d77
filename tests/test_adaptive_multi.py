"""rt_render_adaptive_multi: adaptive sampling with every round's paths spread over the GPUs of one box.

CPU: the argument checks of the entry point on a scene that is not committed, and the exported symbol.
GPU (RTB200_MULTI_ALIAS=1: every logical GPU on the one device, with its own arena, half accumulators, list, stream and workspace):
sums, sample counts, Screen and the path and segment counts equal rt_render (threshold 0) and rt_render_adaptive (above 0) bit for
bit, in every render mode and for GPU counts that do not divide the rounds' paths, also when a round has fewer paths than GPUs and
across call histories that mix GPU counts, image sizes, rt_render_multi and re-commits.  With two or more devices visible the same
runs over real peers."""
import ctypes as C
import os

import numpy as np
import pytest

import ray_tracing_series_rust_b200 as rtb
from ray_tracing_series_rust_b200 import capi
from test_adaptive import ADAPTIVE_CASES

RT_ERR_INVALID, RT_ERR_STATE = -1, -2
FLAGS = {"wavefront": 4, "fused": 8, "pool": 16, "auto": 0}


def _device_count():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


@pytest.fixture
def alias(monkeypatch):
    monkeypatch.setenv("RTB200_MULTI_ALIAS", "1")


# ---------------------------------------------------------------- C-ABI argument checks (no GPU)


@pytest.fixture(scope="module")
def api():
    if not os.path.exists(rtb.LIB_PATH):
        rtb.build()
    api = rtb.load()
    fn = api.lib.rt_render_adaptive_multi
    fn.restype, fn.argtypes = capi.RENDER_ADAPTIVE_MULTI_SIGNATURE
    return api


def _call(api, scene, cfg, ac, n_gpus=2):
    return api.lib.rt_render_adaptive_multi(scene.h if scene is not None else None, C.byref(cfg) if cfg is not None else None,
                                            C.byref(ac) if ac is not None else None, n_gpus, None, None, None, None)


def test_symbol_is_exported():
    assert hasattr(rtb.load().lib, "rt_render_adaptive_multi")


def test_render_adaptive_multi_argument_checks(api):
    s = rtb.new_scene()  # never committed: every rejection below comes from the argument checks
    cfg = capi.make_config(32, 1.0, 16, 5)
    good = dict(min_samples=4, step=2, threshold=0.1, radius=1)

    def ac(**kw):
        d = dict(good)
        d.update(kw)
        return capi.AdaptiveConfig(d["min_samples"], d["step"], d["threshold"], d["radius"])

    bad = [None, ac(step=0), ac(step=-3), ac(threshold=-1e-9), ac(threshold=float("nan")), ac(threshold=float("inf")),
           ac(radius=-1), ac(radius=9), ac(min_samples=-1), ac(min_samples=17)]
    for n in (1, 2, 8):
        for a in bad:
            assert _call(api, s, cfg, a, n) == RT_ERR_INVALID
    for n in (0, -1, 17):
        assert _call(api, s, cfg, ac(), n) == RT_ERR_INVALID
    for flags in ((1 << 16) | (2 << 24), 32):  # RT_RENDER_TILE_SHARD(1, 2), RT_RENDER_NO_WAIT
        assert _call(api, s, capi.make_config(32, 1.0, 16, 5, flags=flags), ac()) == RT_ERR_INVALID
    for s0, s1 in ((1, 0), (0, 8), (2, 16)):
        assert _call(api, s, capi.make_config(32, 1.0, 16, 5, sample_begin=s0, sample_end=s1), ac()) == RT_ERR_INVALID
    assert _call(api, None, cfg, ac()) == RT_ERR_INVALID
    assert _call(api, s, None, ac()) == RT_ERR_INVALID
    assert _call(api, s, cfg, None) == RT_ERR_INVALID
    # valid arguments (the bounds included, mode flags pass through): the scene state is what is wrong
    for n in (1, 2, 16):
        for a, c in ((ac(), cfg), (ac(min_samples=16, radius=8, threshold=0.0, step=1), cfg),
                     (ac(min_samples=0), capi.make_config(32, 1.0, 16, 5, sample_end=16, flags=4 | 2)),
                     (ac(), capi.make_config(32, 1.0, 16, 5, flags=1 << 24))):  # RT_RENDER_TILE_SHARD(0, 1): no sharding
            assert _call(api, s, c, a, n) == RT_ERR_STATE
    s.close()


# ---------------------------------------------------------------- GPU


def _scene(scene_id, param=0, seed=3):
    g = rtb.new_scene()
    g.world_build(scene_id, seed, param)
    g.commit()
    return g


def _assert_same(got, want, what):
    for name, a, b in zip(("screen", "accum", "samples"), got[:3], want[:3]):
        assert np.array_equal(a, b), (what, name)
    assert got[3]["paths"] == want[3]["paths"] and got[3]["segments"] == want[3]["segments"], what


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,param,aspect", [(13, 0, 1.5), (99, 0, 16 / 9), (14, 48, 1.0), (5, 0, 1.0), (6, 0, 1.0)])
def test_threshold_zero_is_rt_render_bit_for_bit(alias, scene_id, param, aspect):
    g = _scene(scene_id, param)
    W, spp = 72, 14
    for mode, flags in FLAGS.items():
        cfg = capi.make_config(W, aspect, spp, 50, seed=4, flags=flags)
        sr, ar, str_ = g.render(cfg, want_accum=True)
        for n in (2, 3, 8):
            sa, aa, smp, sta = g.render_adaptive(cfg, 0.0, min_samples=0, step=3, radius=1, n_gpus=n)
            assert np.array_equal(aa, ar), (mode, n)
            assert np.array_equal(sa, sr), (mode, n)
            assert (smp == spp).all(), (mode, n)
            assert sta["paths"] == str_["paths"] == smp.sum() and sta["segments"] == str_["segments"], (mode, n)
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,aspect,W,spp,min_samples,step,tau,radius,compat", ADAPTIVE_CASES)
def test_adaptive_multi_equals_single_gpu(alias, scene_id, aspect, W, spp, min_samples, step, tau, radius, compat):
    g = _scene(scene_id)
    for mode, flags in FLAGS.items():
        cfg = capi.make_config(W, aspect, spp, 50, seed=6, compat_threads=compat, flags=flags)
        one = g.render_adaptive(cfg, tau, min_samples=min_samples, step=step, radius=radius)
        assert len(np.unique(one[2])) >= 2, "the case must exercise convergence"
        for n in (2, 3, 5):
            _assert_same(g.render_adaptive(cfg, tau, min_samples=min_samples, step=step, radius=radius, n_gpus=n), one, (mode, n))
    g.close()


@pytest.mark.gpu
def test_rounds_with_fewer_paths_than_gpus(alias):
    """6 x 4 pixels, one sample per round, 8 GPUs: once a handful of pixels is left, most GPUs get an empty range"""
    g = _scene(13)
    spp = 40
    cfg = capi.make_config(6, 1.5, spp, 50, seed=5)
    checks = range(2, spp, 2)
    for tau in (0.05, 0.1, 0.2, 0.3, 0.5, 0.8, 1.2, 2.0):
        one = g.render_adaptive(cfg, tau, min_samples=0, step=1, radius=0)
        left = [int((one[2] > c).sum()) for c in checks]  # pixels still active after each check point
        if any(0 < k < 8 for k in left):
            break
    else:
        pytest.fail("no threshold leaves fewer than 8 pixels active")
    for mode, flags in FLAGS.items():
        cfg = capi.make_config(6, 1.5, spp, 50, seed=5, flags=flags)
        _assert_same(g.render_adaptive(cfg, tau, min_samples=0, step=1, radius=0, n_gpus=8),
                     g.render_adaptive(cfg, tau, min_samples=0, step=1, radius=0), (mode, tau))
    g.close()


@pytest.mark.gpu
def test_odd_pixel_count(alias):
    """33 x 33 pixels: W*H*3 is odd, so a replica's B cannot start right after its A (the kernels read A and B with 128-bit loads)"""
    g = _scene(13)
    for mode, flags in FLAGS.items():
        cfg = capi.make_config(33, 1.0, 16, 50, seed=7, flags=flags)
        assert g.image_height(cfg) == 33
        for tau, ms in ((0.0, 0), (0.3, 4)):
            one = g.render_adaptive(cfg, tau, min_samples=ms, step=2, radius=1)
            if tau:
                assert len(np.unique(one[2])) >= 2, "the case must exercise convergence"
            for n in (2, 3):
                _assert_same(g.render_adaptive(cfg, tau, min_samples=ms, step=2, radius=1, n_gpus=n), one, (mode, tau, n))
    g.close()


@pytest.mark.gpu
def test_call_history_sizes_gpu_counts_and_recommits(alias):
    """rt_render_multi, rt_render_adaptive_multi and rt_render_adaptive alternate over two image sizes, 2 -> 4 -> 2 GPUs, a re-commit
    with a new camera and a background change: every result equals its single-GPU counterpart"""
    g = _scene(8, seed=0xB005)
    for f in (0, 30):
        g.set_camera((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, 1.5, 0.1, 10.0, 0.4 * f, 0.4 * f + 0.4)
        g.commit()
        if f:
            g.set_background((0.1, 0.2, 0.9))
        for W in (80, 48):
            cfg = capi.make_config(W, 1.5, 16, 50, seed=4)
            _, a1, _ = g.render(cfg, want_accum=True)
            one = g.render_adaptive(cfg, 0.3, min_samples=4, step=2, radius=1)
            for n in (2, 4, 2):
                _, an, _ = g.render_multi(cfg, n, want_accum=True)
                assert np.array_equal(an, a1), (f, W, n)
                _assert_same(g.render_adaptive(cfg, 0.3, min_samples=4, step=2, radius=1, n_gpus=n), one, (f, W, n))
                _assert_same(g.render_adaptive(cfg, 0.3, min_samples=4, step=2, radius=1), one, (f, W, n))
    g.close()


@pytest.mark.gpu
def test_python_entry_point(alias):
    g = _scene(13)
    cfg = capi.make_config(40, 1.5, 12, 20, seed=2)
    one = g.render_adaptive(cfg, 0.3, min_samples=0, step=2, radius=1, n_gpus=1)
    three = g.render_adaptive(cfg, 0.3, min_samples=0, step=2, radius=1, n_gpus=3)
    assert [a.shape for a in three[:3]] == [a.shape for a in one[:3]] and three[2].dtype == np.int32
    _assert_same(three, one, "n_gpus=3")
    with pytest.raises(capi.RtError) as e:
        g.render_adaptive(cfg, 0.3, n_gpus=0)
    assert e.value.code == RT_ERR_INVALID
    g.close()


@pytest.mark.gpu
@pytest.mark.skipif(_device_count() < 2, reason="needs two visible GPUs")
def test_adaptive_multi_over_real_peers(monkeypatch):
    """no alias: GPU 0 reads the other GPUs' half accumulators over NVLink and copies them each new list"""
    monkeypatch.delenv("RTB200_MULTI_ALIAS", raising=False)
    n_dev = _device_count()
    for case, flags in ((ADAPTIVE_CASES[0], 0), (ADAPTIVE_CASES[4], 4)):  # book-1 (fused), scene 6 (wavefront on every GPU)
        scene_id, aspect, W, spp, min_samples, step, tau, radius, compat = case
        g = _scene(scene_id)
        cfg = capi.make_config(W, aspect, spp, 50, seed=6, compat_threads=compat, flags=flags)
        one = g.render_adaptive(cfg, tau, min_samples=min_samples, step=step, radius=radius)
        assert len(np.unique(one[2])) >= 2
        for n in sorted({2, n_dev}):
            _assert_same(g.render_adaptive(cfg, tau, min_samples=min_samples, step=step, radius=radius, n_gpus=n), one, (scene_id, n))
        g.close()
