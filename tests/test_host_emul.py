"""The device functions of csrc/cuda/rt_device.cuh, compiled for the HOST (tests/host_emul, g++ + a small CUDA shim), run
over the host-flattened scene arrays (rt_debug_host_scene) and are compared with the oracle on the E1 ray batches.

This is what a machine without a GPU can say about the device code itself: the flattener, both BVH layouts (sibling
pairs and the 4-wide collapse), the f32 slab tests, the f64 primitive tests, transforms and hit records are the very
source the kernels compile — only the SIMT execution differs (a "warp" is one lane here).  Test infrastructure only:
the product has no CPU path (test_commit_fails_loudly_without_gpu).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import ray_tracing_series_rust_b200 as rtb
from ray_tracing_series_rust_b200 import capi

import parity_utils as pu

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_emul")


def _build_emul(so, extra=()):
    """Compiles emul.cpp to `so`, a fresh path of this test session: a library kept between sessions could predate a change to
    any header emul.cpp includes, and parallel test workers must not write one file at once."""
    cuda_include = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", *extra,
                           "-I" + cuda_include, os.path.join(HERE, "emul.cpp"), "-o", so])
    lib = C.CDLL(so)
    lib.emul_sizeof_device_scene.restype = C.c_uint64
    lib.emul_trace_batch.restype = C.c_int32
    lib.emul_trace_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_int32, C.c_uint64, C.c_int32, C.c_void_p, C.c_void_p]
    lib.emul_trace_wide.restype = C.c_int32
    lib.emul_trace_wide.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_double, C.c_int32, C.c_int32, C.c_void_p]
    lib.emul_render.restype = C.c_int32
    lib.emul_render.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_int32, C.c_void_p, C.c_void_p]
    if not os.path.exists(rtb.LIB_PATH):
        rtb.build()
    return lib


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    return _build_emul(str(tmp_path_factory.mktemp("emul") / "libemul.so"))


def host_scene(emul, scene_id, seed=0xB001, param=0, width=2):
    s = rtb.new_scene()
    s.world_build(scene_id, seed, param)
    s.set_bvh_width(width)
    return s, s.debug_host_scene(emul.emul_sizeof_device_scene())


def emul_trace(emul, dscene, rays, t_min=0.001, t_max=float("inf"), flags=capi.RT_TRACE_SKIP_MEDIA, seed=0, wide=0, counts=None):
    rays = np.ascontiguousarray(rays, dtype=capi.RAY_DTYPE)
    out = np.zeros(rays.shape[0], dtype=capi.HIT_DTYPE)
    cnt = (C.c_uint64 * 2)()
    assert emul.emul_trace_batch(dscene, rays.ctypes.data, rays.shape[0], t_min, t_max, flags, seed, wide, out.ctypes.data, cnt) == 0
    if counts is not None:
        counts.update(boxes=int(cnt[0]), prims=int(cnt[1]))
    return out


def emul_trace_wide(emul, dscene, rays, resume, t_min=0.001, t_max=float("inf"), pm3=0):
    rays = np.ascontiguousarray(rays, dtype=capi.RAY_DTYPE)
    out = np.zeros(rays.shape[0], dtype=capi.HIT_DTYPE)
    assert emul.emul_trace_wide(dscene, rays.ctypes.data, rays.shape[0], t_min, t_max, resume, pm3, out.ctypes.data) == 0
    return out


def oracle_scene(orc, scene_id, seed=0xB001, param=0):
    o = orc.new_scene()
    o.world_build(scene_id, seed, param)
    o.commit()
    return o


# id: (box lo, box hi, allowed id-mismatch fraction, allowed tie fraction) — the bounds of tests/test_gpu_parity.py
SCENES = {
    13: (-15.0, 15.0, 0.0, 0.0),
    99: (-15.0, 15.0, 0.0, 0.0),
    4: (0.0, 555.0, 0.0, 0.0),
    5: (0.0, 555.0, 0.0, 0.0),
    6: (-600.0, 600.0, 0.0, 0.02),
    8: (-15.0, 15.0, 0.0, 0.0),
    14: (-30.0, 56.0, 2e-4, 0.0),
}


@pytest.mark.parametrize("scene_id", sorted(SCENES))
def test_device_functions_on_host_match_the_oracle(orc, emul, scene_id):
    lo, hi, frac, ties = SCENES[scene_id]
    param = 32 if scene_id == 14 else 0
    s, ds = host_scene(emul, scene_id, param=param)
    o = oracle_scene(orc, scene_id, param=param)
    cam = pu.camera_fields(orc, o)
    tr = (cam["time1"], cam["time2"])
    tfrac = 1e-3 if scene_id == 14 else 0.0
    for name, rays in (("primary", pu.primary_rays(cam, 96, 54)), ("random", pu.random_rays(12000, lo, hi, seed=scene_id + 1, time_range=tr))):
        he, ho = emul_trace(emul, ds, rays), o.trace_batch(rays)
        pu.assert_parity(he, ho, f"emul scene {scene_id} {name}", max_id_frac=frac, max_tie_frac=ties, max_t_frac=tfrac, rays=rays)
        sec = pu.secondary_rays(ho, seed=7, time=0.5 * (tr[0] + tr[1]))
        if sec.shape[0]:
            pu.assert_parity(emul_trace(emul, ds, sec), o.trace_batch(sec), f"emul scene {scene_id} {name} secondary", max_id_frac=max(frac, 2e-5),
                             max_tie_frac=ties, max_t_frac=tfrac, rays=sec, require_hits=False)
    s.close()
    o.close()


@pytest.mark.parametrize("scene_id,param", [(14, 32), (14, 96), (14, 260), (13, 0), (10, 0)])  # 14/260: 135 200 triangles, the parallel collapse
def test_wide_walk_equals_pair_walk(orc, emul, scene_id, param):
    """The 4-wide collapse (bvh_wide.hpp) + trace_wide return the SAME hit records, bit for bit, as the sibling-pair walk:
    closest hit is topology independent and exact ties are decided by depth-first id, not by visiting order."""
    s2, d2 = host_scene(emul, scene_id, param=param, width=2)
    s4, d4 = host_scene(emul, scene_id, param=param, width=4)
    lo, hi = (-30.0, 56.0) if scene_id == 14 else (-15.0, 15.0)
    o = oracle_scene(orc, scene_id, param=param)
    cam = pu.camera_fields(orc, o)
    batches = [pu.primary_rays(cam, 128, 72), pu.random_rays(20000, lo, hi, seed=11, time_range=(cam["time1"], cam["time2"]))]
    batches.append(pu.secondary_rays(o.trace_batch(batches[0]), seed=3, time=cam["time1"]))
    n_hits = 0
    for rays in batches:
        ref = emul_trace(emul, d2, rays)
        for resume in (0, 1):
            w = emul_trace_wide(emul, d4, rays, resume)
            assert w.tobytes() == ref.tobytes(), (scene_id, resume, int((w["prim_id"] != ref["prim_id"]).sum()))
        n_hits += int((ref["prim_id"] >= 0).sum())
    assert n_hits > 1000
    for x in (s2, s4, o):
        x.close()


@pytest.mark.parametrize("scene_id", [4, 5, 6, 8, 13, 14, 99])
def test_wide_world_hit_equals_pair_world_hit(orc, emul, scene_id):
    """world_hit<..., WIDE> (what k_extend<..., WIDE> runs when rt_scene_set_bvh_width(4) forces it): every main-world instance
    through its own 4-wide root, wrappers and media (pair-walked boundaries, seeded draws) included: identical hit records."""
    param = 32 if scene_id == 14 else 0
    s2, d2 = host_scene(emul, scene_id, param=param, width=2)
    s4, d4 = host_scene(emul, scene_id, param=param, width=4)
    o = oracle_scene(orc, scene_id, param=param)
    cam = pu.camera_fields(orc, o)
    lo, hi = SCENES[scene_id][:2]
    prim = pu.primary_rays(cam, 120, 68)
    batches = [prim, pu.random_rays(15000, lo, hi, seed=5, time_range=(cam["time1"], cam["time2"])), pu.secondary_rays(o.trace_batch(prim), seed=3, time=cam["time1"])]
    for rays in batches:
        for flags in (capi.RT_TRACE_SKIP_MEDIA, capi.RT_TRACE_SEEDED_MEDIA):
            c2, c4 = {}, {}
            ref = emul_trace(emul, d2, rays, flags=flags, seed=17, counts=c2)
            w = emul_trace(emul, d4, rays, flags=flags, seed=17, wide=1, counts=c4)
            assert w.tobytes() == ref.tobytes(), (scene_id, flags, int((w["prim_id"] != ref["prim_id"]).sum()))
            assert c4["prims"] <= 1.05 * c2["prims"]  # queued leaves behind closest_so_far are dropped (the queued children are not sorted: a few more than the ordered pair walk on some scenes)
    for x in (s2, s4, o):
        x.close()


def test_wide_collapse_is_built_only_where_asked_or_measured(emul):
    nbytes = emul.emul_sizeof_device_scene()
    for scene_id, width, built in ((5, 0, True), (6, 0, True), (5, 2, False), (3, 0, False), (8, 0, True), (99, 0, True), (8, 2, False), (13, 0, True), (13, 2, False), (6, 4, True), (5, 4, True)):
        s, ds = host_scene(emul, scene_id, width=width)
        assert (emul.emul_trace_batch(ds, None, 0, 0.001, 1.0, 0, 0, 1, None, None) == 0) == built, (scene_id, width)
        s.close()
    s = rtb.new_scene()
    with pytest.raises(Exception):
        s.set_bvh_width(3)
    with pytest.raises(Exception):
        s.debug_host_scene(nbytes - 8)
    s.close()


def test_wide_collapse_edge_cases(orc, emul, monkeypatch):
    """Root that is a single leaf, two primitives, a degenerate (empty) world, leaves too large for a wide reference."""
    nbytes = emul.emul_sizeof_device_scene()

    def build(s, n):
        m = s.lambertian((0.5, 0.5, 0.5))
        objs = [s.sphere((2.5 * i, 0.3 * i, -1.0 * i), 1.0, m) for i in range(n)]
        s.set_root(s.bvh(objs, 0, 1) if n else s.list([]))
        s.set_camera((0, 1, 12), (0, 0, 0), (0, 1, 0), 40, 1.5, 0.0, 10, 0, 1)

    for n in (1, 2, 3, 5, 9):
        g, o = rtb.new_scene(), orc.new_scene()
        build(g, n); build(o, n)
        o.commit()
        g.set_bvh_width(4)
        ds = g.debug_host_scene(nbytes)
        rays = np.concatenate([pu.random_rays(8000, -3.0, 3.0 * n, seed=n), pu.primary_rays(pu.camera_fields(orc, o), 150, 100)])
        ho = o.trace_batch(rays)
        assert (ho["prim_id"] >= 0).sum() > 100
        pu.assert_parity(emul_trace(emul, ds, rays, wide=1), ho, f"{n} spheres wide")
        assert emul_trace_wide(emul, ds, rays, 0).tobytes() == emul_trace(emul, ds, rays).tobytes()
        g.close(); o.close()
    g = rtb.new_scene()
    build(g, 0)
    g.set_bvh_width(4)
    ds = g.debug_host_scene(nbytes)  # no instances: nothing to collapse, pair and wide entry both see an empty world
    rays = pu.random_rays(16, -1.0, 1.0, seed=1)
    assert (emul_trace(emul, ds, rays)["prim_id"] == -1).all()
    g.close()
    monkeypatch.setenv("RTB200_MAX_LEAF", "16")  # larger leaves: a leaf of > 8 primitives would not fit a wide reference (the scene then stays on pairs)
    g = rtb.new_scene()
    g.world_build(13, 0xB001, 0)
    g.set_bvh_width(4)
    ds = g.debug_host_scene(nbytes)
    rays = pu.random_rays(6000, -15.0, 15.0, seed=2)
    ref = emul_trace(emul, ds, rays)
    if emul.emul_trace_batch(ds, None, 0, 0.001, 1.0, 0, 0, 1, None, None) == 0:
        assert emul_trace(emul, ds, rays, wide=1).tobytes() == ref.tobytes()
    assert (ref["prim_id"] >= 0).sum() > 500
    g.close()


def emul_render(emul, dscene, W, H, spp, depth, seed, wide=0, sample_begin=0, sample_end=None):
    acc = np.zeros((H, W, 3), dtype=np.int64)
    seg = C.c_uint64(0)
    assert emul.emul_render(dscene, W, H, spp, sample_begin, spp if sample_end is None else sample_end, depth, seed, wide, acc.ctypes.data, C.byref(seg)) == 0
    return acc, int(seg.value)


@pytest.mark.parametrize("scene_id,W,aspect,spp", [(13, 60, 1.5, 6), (99, 60, 16 / 9, 6), (4, 40, 1.0, 8), (5, 40, 1.0, 8), (6, 40, 1.0, 6), (8, 60, 1.5, 4), (14, 40, 1.0, 6),
                                                   (1, 40, 1.5, 4), (2, 40, 1.5, 4), (3, 40, 1.5, 6)])
def test_device_path_loop_on_host_matches_the_oracle_sample_by_sample(orc, emul, scene_id, W, aspect, spp):
    """E2 without a GPU: camera_first_ray, world_hit, every Material::scatter / Texture::value / Perlin and the fixed-point
    accumulation of the DEVICE header, run path by path on the host with the kernels' Philox streams, against the oracle's
    int64 sums (same bars as tests/test_gpu_parity.py::test_E2_render_matches_oracle_sample_by_sample)."""
    param = 32 if scene_id == 14 else 0
    s, ds = host_scene(emul, scene_id, param=param, width=4 if scene_id in (6, 13) else 2)
    o = oracle_scene(orc, scene_id, param=param)
    cfg = capi.make_config(W, aspect, spp, 50, seed=21)
    so, ao, sto = o.render(cfg, want_accum=True)
    H = ao.shape[0]
    ae, seg = emul_render(emul, ds, W, H, spp, 50, 21, wide=1 if scene_id in (6, 13) else 0)
    fe, fo = ae / capi.ACCUM_SCALE, ao / capi.ACCUM_SCALE
    rel = np.abs(fe - fo) / np.maximum(1e-3, np.abs(fo))
    pix_bad = (rel > 1e-5).any(axis=2)
    assert pix_bad.mean() < 0.02, (pix_bad.mean(), seg, sto["segments"])
    assert abs(fe.mean() - fo.mean()) <= 0.01 * max(fo.mean(), 1e-3)
    assert abs(seg - sto["segments"]) <= 0.005 * sto["segments"]
    # sample ranges add up exactly (integer sums, streams keyed by the global sample index): the sharding contract
    a0, _ = emul_render(emul, ds, W, H, spp, 50, 21, wide=1 if scene_id in (6, 13) else 0, sample_begin=0, sample_end=spp // 2)
    a1, _ = emul_render(emul, ds, W, H, spp, 50, 21, wide=1 if scene_id in (6, 13) else 0, sample_begin=spp // 2, sample_end=spp)
    assert np.array_equal(a0 + a1, ae)
    s.close()
    o.close()


@pytest.mark.parametrize("scene_id", [99, 7])
def test_motion_form_of_the_wide_walk(orc, emul, scene_id):
    """MovingSphere scenes (book-1 as shipped, the moving-sphere test scene): trace_wide<spheres + moving spheres> interpolates
    the child boxes of DeviceScene::mnodes4 at the ray's time; hits equal the pair walk over union boxes, bit for bit, at
    shutter start, end, in between and (clamped) outside."""
    s2, d2 = host_scene(emul, scene_id, width=2)
    s4, d4 = host_scene(emul, scene_id, width=4)
    o = oracle_scene(orc, scene_id)
    cam = pu.camera_fields(orc, o)
    t1, t2 = cam["time1"], cam["time2"]
    n_hits = 0
    for time in (t1, t2, 0.5 * (t1 + t2), t1 + 0.123 * (t2 - t1)):
        prim = pu.primary_rays(cam, 120, 68, time=time)
        for rays in (prim, pu.secondary_rays(o.trace_batch(prim), seed=9, time=time)):
            ref = emul_trace(emul, d2, rays)
            pu.assert_parity(ref, o.trace_batch(rays), f"scene {scene_id} t={time}", require_hits=False)
            for resume in (0, 1):
                w = emul_trace_wide(emul, d4, rays, resume, pm3=1)
                assert w.tobytes() == ref.tobytes(), (scene_id, time, resume, int((w["prim_id"] != ref["prim_id"]).sum()))
            n_hits += int((ref["prim_id"] >= 0).sum())
    rnd = pu.random_rays(8000, -15.0, 15.0, seed=6, time_range=(t1, t2))
    assert emul_trace_wide(emul, d4, rnd, 0, pm3=1).tobytes() == emul_trace(emul, d2, rnd).tobytes()
    assert n_hits > 5000
    s13, d13 = host_scene(emul, 13, width=4)  # no moving spheres: no motion form
    assert emul.emul_trace_wide(d13, None, 0, 0.001, 1.0, 0, 1, None) == -2
    for x in (s2, s4, o, s13):
        x.close()


def test_rng_conversions_equal_the_formulas_they_replace(emul):
    """PathRng::unit_of / pm1_of (bits of 2^52 + u, one fma) against (double)u * 2^-32 and fma(xi, 2, -1): bit-equal for the edge
    words and 2 M random ones (both forms are exact, so this is an identity, not a tolerance)."""
    emul.emul_rng_convert_mismatches.restype = C.c_uint64
    emul.emul_rng_convert_mismatches.argtypes = [C.c_uint64, C.c_uint64]
    assert emul.emul_rng_convert_mismatches(2_000_000, 0x9E3779B97F4A7C15) == 0


@pytest.mark.parametrize("scene_id,param,W,H,spp,max_index", [(13, 0, 120, 80, 2, 12), (14, 64, 60, 60, 2, 32)])
def test_wide_stack_depth_stays_far_below_its_capacity(emul, scene_id, param, W, H, spp, max_index):
    """The 4-wide walk's stack (RT_WIDE_STACK = 96 entries per lane) as the fused kernels use it: accesses per index over whole
    paths.  book-1 never goes past 8 entries (the full 871 200-triangle mesh: 19, tools/ measured once); what the shared-memory
    stack experiment of round 2 was sized with (profiles/r2_50_ab_signed_rows_smem_stack.txt)."""
    emul.emul_wide_stack_hist.restype = C.c_int32
    emul.emul_wide_stack_hist.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_void_p, C.c_void_p]
    s, ds = host_scene(emul, scene_id, param=param, width=4)
    hist = np.zeros(96, dtype=np.uint64)
    seg = C.c_uint64(0)
    assert emul.emul_wide_stack_hist(ds, W, H, spp, 50, 3, hist.ctypes.data, C.byref(seg)) == 0
    assert seg.value > W * H * spp and hist.sum() > 0
    assert int(np.nonzero(hist)[0].max()) < max_index
    s.close()


@pytest.mark.parametrize("scene_id,param,W,H,spp", [(13, 0, 60, 40, 6), (99, 0, 64, 36, 4), (6, 0, 40, 40, 4), (5, 0, 40, 40, 6), (14, 32, 40, 40, 4), (1, 0, 48, 32, 4)])
def test_fused_order_of_shading_draws_the_same_numbers(emul, scene_id, param, W, H, spp):
    """The fused kernels open the scatter event before the branch on the material and run one rejection loop for Lambertian, Metal
    and Isotropic lanes (lambertian_finish / metal_finish / isotropic_finish); k_shade_all calls scatter_* per material.  Same draws
    in the same order: the two orders give the same int64 sums, bit for bit (on the GPU: test_fused_mode_is_bit_identical_to_wavefront)."""
    s, ds = host_scene(emul, scene_id, param=param, width=2)
    a0, s0 = emul_render(emul, ds, W, H, spp, 50, 33, wide=0)
    a1, s1 = emul_render(emul, ds, W, H, spp, 50, 33, wide=2)
    assert s0 == s1 and np.array_equal(a0, a1)
    s.close()


def test_multi_draw_samplers_equal_single_draws_from_any_position(emul):
    """next3_pm1 / next2_pm1 (three / two words at once, picked with selects, at most one new Philox block) against single
    gen_range(-1, 1) draws, from every draw position 0..23, with the start block cached or not, interleaved with single draws:
    same doubles, same draw counter.  Covers the positions the renders never reach (their events start on block boundaries)."""
    emul.emul_rng_multi_draw_mismatches.restype = C.c_uint64
    emul.emul_rng_multi_draw_mismatches.argtypes = [C.c_uint64, C.c_uint64]
    assert emul.emul_rng_multi_draw_mismatches(0xB200, 200) == 0
