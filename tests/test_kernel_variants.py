"""Every render kernel launch_render can launch (csrc/cuda/kernels.cu), each reached through a scene, knobs and render flags.

launch_render picks one of the k_extend / k_extend_p / k_mega / k_mega_r / k_pool template instances from the scene's properties
(primitive mask, wrappers, media, 4-wide tree, large meshes), the render flags and the knobs read at rt_scene_create.  The
instances compile different code, so a wrong choice or a bug in one instance shows only in the scenes that reach it.

VARIANTS holds one row per instance: the kernel with its template arguments, and the ways to reach it.
- CPU: every instance in the ptxas log (csrc/build/kernels.ptxas.log) is claimed by exactly one row.
- GPU: for every way, the kernel that ran (torch.profiler) is the row's kernel.  Its accumulator and segment count equal the
  forced-wavefront render of the same scene with default knobs (forced fused for wavefront kernels).  The oracle's render of the
  same paths meets the sample-by-sample bar of test_E2_render_matches_oracle_sample_by_sample.
- GPU, per kernel family: renders of 1, 31, 33 and 129 paths and a render one path past a multiple of 32 (the claim unit of the
  persistent kernels); path ids (pixel * spp + sample) past 2^32; sample-major enumeration indices past 2^32 and 2^33; and one
  render of more than 2^32 paths against its closed form.
"""
import ctypes as C
import os
import re
import time
from collections import namedtuple

import numpy as np
import pytest

import ray_tracing_series_rust_b200 as rtb
from ray_tracing_series_rust_b200 import capi

LOG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ray_tracing_series_rust_b200", "csrc", "build",
                   "kernels.ptxas.log")
RENDER_KERNELS = ("k_extend", "k_extend_p", "k_mega", "k_mega_r", "k_pool")

COUNT, WAVE, FUSED, POOL = 2, 4, 8, 16  # RT_RENDER_COUNT_EVENTS, _FORCE_WAVEFRONT, _FORCE_FUSED, _FORCE_POOL
SPEC0, SPEC1 = (("RTB200_PRIM_SPECIALISE", "0"),), (("RTB200_PRIM_SPECIALISE", "1"),)
WAIT0, WAIT16 = (("RTB200_MEGA_WAIT", "0"),), (("RTB200_MEGA_WAIT", "16"),)


# ---------------------------------------------------------------- kernel names -> (name, template arguments...)
def decode_kernel(name):
    """A render kernel's name, mangled (_ZN3rtb6k_megaILb0ELi6E...) or demangled (void rtb::k_mega<false, 6, ...>(...)), as
    (name, arg, ...) with bool and int arguments; None for any other kernel."""
    m = re.match(r"_ZN3rtb(\d+)", name)
    if m:
        n = int(m.group(1))
        kname, rest = name[m.end():m.end() + n], name[m.end() + n:]
        targs = re.match(r"I((?:L[bij]n?\d+E)+)E", rest)
        if kname not in RENDER_KERNELS or not targs:
            return None
        args = [bool(int(v)) if t == "b" else int(v.replace("n", "-")) for t, v in re.findall(r"L([bij])(n?\d+)E", targs.group(1))]
        return (kname, *args)
    m = re.search(r"rtb::(k_\w+)<([^<>]*)>", name)
    if not m or m.group(1) not in RENDER_KERNELS:
        return None
    args = []
    for a in m.group(2).split(","):
        a = a.strip()
        args.append(a == "true" if a in ("true", "false") else int(a.rstrip("u")))
    return (m.group(1), *args)


def cxx(kernel):
    return kernel[0] + "<" + ",".join(("true" if a else "false") if isinstance(a, bool) else str(a) for a in kernel[1:]) + ">"


def log_instances():
    text = open(LOG).read()
    syms = set(re.findall(r"Function properties for (_ZN3rtb\d+k_\w+I\S+)", text))
    return {k for k in map(decode_kernel, syms) if k is not None}


# ---------------------------------------------------------------- scenes built identically in the product and the oracle
def wrapped_spheres(s):
    """book-1 style: ground, three large spheres and small spheres, partly under Translate / RotateY"""
    ground = s.sphere((0, -1000, 0), 1000, s.lambertian((0.5, 0.5, 0.5)))
    mats = [s.lambertian((0.8, 0.3, 0.2)), s.metal((0.7, 0.6, 0.5), 0.1), s.dielectric(1.5), s.lambertian((0.2, 0.4, 0.8))]
    small = [s.sphere((0.9 * a, 0.2, 0.9 * b), 0.2, mats[(a * 7 + b) % 4]) for a in range(-5, 6) for b in range(-5, 6) if (a + b) % 2 == 0]
    big = [s.sphere((0, 1, 0), 1.0, mats[2]), s.sphere((-4, 1, 0), 1.0, mats[0]), s.sphere((4, 1, 0), 1.0, mats[1])]
    s.set_root(s.list([ground, s.translate((0.3, 0, -0.2), s.rotate_y(20, s.bvh(small, 0, 1))), s.translate((0, 0.1, 0), s.list(big))]))
    s.set_camera((13, 2, 3), (0, 0, 0), (0, 1, 0), 20, 1.5, 0.1, 10, 0, 1)
    s.set_background((0.7, 0.8, 1.0))


def wrapped_moving(s):
    """moving spheres (and a static ground) under a Translate"""
    ground = s.sphere((0, -1000, 0), 1000, s.lambertian((0.5, 0.6, 0.5)))
    mats = [s.lambertian((0.8, 0.3, 0.2)), s.metal((0.7, 0.6, 0.5), 0.2), s.dielectric(1.5)]
    balls = [s.moving_sphere((a, 0.3, b), (a, 0.3 + 0.1 * ((a + b) % 3), b), 0, 1, 0.3, mats[(a + 2 * b) % 3])
             for a in range(-4, 5) for b in range(-3, 4)]
    s.set_root(s.list([ground, s.translate((0.2, 0, 0.1), s.bvh(balls, 0, 1))]))
    s.set_camera((13, 2, 3), (0, 0, 0), (0, 1, 0), 20, 1.5, 0.1, 10, 0, 1)
    s.set_background((0.7, 0.8, 1.0))


def _grid_mesh(n):
    """a bumpy n x n height field: 2 n^2 triangles"""
    x, z = np.meshgrid(np.linspace(-200.0, 200.0, n + 1), np.linspace(-200.0, 200.0, n + 1))
    y = 60.0 + 25.0 * np.sin(x / 37.0) * np.cos(z / 29.0)
    verts = np.stack([x, y, z], axis=-1).reshape(-1, 3)
    i, j = np.meshgrid(np.arange(n), np.arange(n))
    a = (j * (n + 1) + i).reshape(-1)
    b, c, d = a + 1, a + n + 1, a + n + 2
    return verts, np.concatenate([np.stack([a, b, c], 1), np.stack([b, d, c], 1)])


def wrapped_mesh(s):
    """4608 triangles and rects (floor, back wall, light) under a Translate: the wavefront takes k_extend_p through an instance chain"""
    verts, idx = _grid_mesh(48)
    white, red = s.lambertian((0.73, 0.73, 0.73)), s.lambertian((0.65, 0.05, 0.05))
    mesh = s.triangle_mesh(verts, idx, red)
    room = s.list([s.xz_rect(-300, 300, -300, 300, 0, white), s.xy_rect(-300, 300, 0, 300, 250, white),
                   s.xz_rect(-80, 80, -80, 80, 299, s.diffuse_light((7, 7, 7)))])
    s.set_root(s.translate((10, 0, -5), s.list([s.bvh([mesh], 0, 1), room])))
    s.set_camera((0, 200, -500), (0, 60, 0), (0, 1, 0), 50, 1.0, 0.0, 10, 0, 1)
    s.set_background((0.1, 0.1, 0.15))


def _textured(s, moving, image):
    if image:
        u, v = np.meshgrid(np.arange(32), np.arange(16))
        tex = s.tex_image(np.stack([u * 8, v * 16, (u + v) * 5 % 256], axis=-1).astype(np.float64))
    else:
        tex = s.tex_noise(2.0, seed=11)
    mats = [s.lambertian(tex), s.metal((0.7, 0.6, 0.5), 0.1), s.dielectric(1.5), s.lambertian((0.3, 0.5, 0.2))]
    if moving:
        prims = [s.sphere((0, -1000, 0), 1000, mats[0])]
        prims += [s.moving_sphere((a, 0.4, b), (a, 0.4 + 0.2 * ((a * b) % 2), b), 0, 1, 0.4, mats[(a + b) % 4]) for a in range(-3, 4) for b in range(-2, 3)]
    else:
        prims = [s.sphere((0, -1000, 0), 1000, mats[0])]
        prims += [s.gravity_sphere((a, 0.5 + 0.3 * ((a + b) % 3), b), 0.0, 0.4, mats[(a + b) % 4]) for a in range(-3, 4) for b in range(-2, 3)]
    s.set_root(s.bvh(prims, 0, 1))
    s.set_camera((13, 2, 3), (0, 0, 0), (0, 1, 0), 20, 1.5, 0.0, 10, 0, 1)
    s.set_background((0.7, 0.8, 1.0))


def moving_noise(s): _textured(s, True, False)
def moving_image(s): _textured(s, True, True)
def gravity_noise(s): _textured(s, False, False)
def gravity_image(s): _textured(s, False, True)


def medium_and_triangles(s):
    """a ConstantMedium with a one-sphere boundary next to a triangle mesh: media plus a primitive mask outside 0x1b"""
    verts, idx = _grid_mesh(6)
    white = s.lambertian((0.73, 0.73, 0.73))
    mesh = s.triangle_mesh(verts * (0.5, 1.0, 0.5), idx, s.lambertian((0.2, 0.6, 0.3)))
    fog = s.constant_medium((0.9, 0.9, 0.9), 0.01, s.sphere((0, 100, 0), 80, white))
    s.set_root(s.list([s.bvh([mesh], 0, 1), fog, s.xz_rect(-300, 300, -300, 300, 0, white),
                       s.xz_rect(-60, 60, -60, 60, 290, s.diffuse_light((10, 10, 10)))]))
    s.set_camera((0, 150, -400), (0, 80, 0), (0, 1, 0), 50, 1.0, 0.0, 10, 0, 1)
    s.set_background((0.05, 0.05, 0.08))


def general_medium(s):
    """wrapper chains, a shared group and a medium whose boundary is a list of two spheres (no one-sphere / one-box fast path)"""
    m = s.lambertian((0.5, 0.5, 0.5))
    sph = s.sphere((0, 0, 0), 1.0, s.dielectric(1.5))
    box = s.box((-1, -1, -1), (1, 2, 1.5), m)
    tri = s.triangle((0, 0, 0), (2, 0, 0.5), (0, 2, 1), m)
    group = s.list([sph, s.translate((3, 0, 0), box)])
    med = s.constant_medium((1, 1, 1), 0.3, s.list([s.sphere((0, 0, -8), 2.0, m), s.sphere((1, 0, -8), 2.0, m)]))
    s.set_root(s.list([s.translate((-6, 0, 0), s.rotate_y(30, s.translate((0, 1, 0), group))), s.rotate_y(-50, s.list([box, tri])),
                       s.translate((6, 0, 2), group), med]))
    s.set_camera((0, 3, 25), (0, 0, 0), (0, 1, 0), 40, 1.5, 0.0, 10, 0, 1)
    s.set_background((0.7, 0.8, 1.0))


MESH = (14, 48)  # the mesh room at 4608 triangles: a large mesh (>= 4096 triangles) in one wrapper-free instance
ASPECT = {13: 1.5, 99: 16 / 9, 8: 1.5, 2: 16 / 9, wrapped_spheres: 1.5, wrapped_moving: 1.5, moving_noise: 1.5, moving_image: 1.5,
          gravity_noise: 1.5, gravity_image: 1.5, general_medium: 1.5}


def aspect_of(scene):
    return ASPECT.get(scene[0] if isinstance(scene, tuple) else scene, 1.0)


def scene_name(scene):
    return f"s{scene[0]}" + (f"p{scene[1]}" if scene[1] else "") if isinstance(scene, tuple) else scene.__name__


def build(scene, s, width=0):
    """Build and commit `scene` ((world id, param) or a builder function) into s; width: rt_scene_set_bvh_width (product only)."""
    if isinstance(scene, tuple):
        s.world_build(scene[0], 0xB001, scene[1])
    else:
        scene(s)
    if width:
        s.set_bvh_width(width)
    return s.commit()


# ---------------------------------------------------------------- the table
Way = namedtuple("Way", "scene flags width env", defaults=(0, ()))
F, T = False, True

VARIANTS = [
    # k_extend<MEDIA, COUNT, MINB, GENERAL_MEDIA, PM, WIDE>: the wavefront's one-ray-per-thread extend kernel
    (("k_extend", F, F, 5, F, 63, F), [Way((13, 0), WAVE)]),
    (("k_extend", F, T, 4, F, 63, F), [Way((4, 0), COUNT)]),  # Cornell box: wrappers, so no 4-wide tree
    (("k_extend", F, T, 4, F, 63, T), [Way((13, 0), COUNT)]),  # the counting pass walks the tree the fused kernel walks
    (("k_extend", T, F, 4, F, 63, F), [Way(medium_and_triangles, WAVE), Way((5, 0), WAVE, 0, SPEC0)]),
    (("k_extend", T, F, 4, T, 63, F), [Way(general_medium, WAVE)]),
    (("k_extend", T, F, 5, F, 24, F), [Way((5, 0), WAVE, 2)]),
    (("k_extend", T, F, 5, F, 24, T), [Way((5, 0), WAVE)]),
    (("k_extend", T, F, 5, F, 27, F), [Way((6, 0), WAVE, 2)]),
    (("k_extend", T, F, 5, F, 27, T), [Way((6, 0), WAVE)]),
    (("k_extend", T, T, 4, F, 63, F), [Way((5, 0), COUNT), Way((6, 0), COUNT)]),
    (("k_extend", T, T, 4, T, 63, F), [Way(general_medium, COUNT)]),
    # k_extend_p<MEDIA, COUNT, MINB>: the persistent warp-scheduled extend kernel of large meshes
    (("k_extend_p", F, F, 4), [Way(wrapped_mesh, WAVE), Way(MESH, WAVE)]),
    (("k_extend_p", F, T, 4), [Way(MESH, COUNT, 2)]),
    # k_mega<MEDIA, MINB, GENERAL_MEDIA, PM, XF, WIDE, FULLTEX>: the fused persistent kernel
    (("k_mega", F, 4, F, 1, T, F, T), [Way(wrapped_spheres, FUSED), Way((13, 0), FUSED, 0, SPEC1)]),
    (("k_mega", F, 4, F, 3, T, F, T), [Way(wrapped_moving, FUSED)]),
    (("k_mega", F, 4, F, 40, T, F, T), [Way(wrapped_mesh, FUSED), Way(MESH, FUSED, 0, SPEC1)]),
    (("k_mega", F, 4, F, 63, T, F, T), [Way((13, 0), FUSED, 0, SPEC0), Way(MESH, FUSED, 0, SPEC0)]),
    (("k_mega", F, 5, F, 1, F, F, T), [Way((13, 0), FUSED, 2)]),
    (("k_mega", F, 5, F, 1, F, T, T), [Way((2, 0), FUSED)]),  # image texture on the 4-wide tree
    (("k_mega", F, 5, F, 3, F, F, T), [Way((99, 0), FUSED, 2)]),
    (("k_mega", F, 5, F, 3, F, T, T), [Way(moving_noise, FUSED, 4), Way(moving_image, FUSED, 4)]),
    (("k_mega", F, 5, F, 5, F, F, T), [Way((8, 0), FUSED, 0, WAIT16), Way((8, 0), FUSED, 2)]),
    (("k_mega", F, 5, F, 5, F, T, T), [Way(gravity_noise, FUSED, 4), Way(gravity_image, FUSED, 4)]),
    (("k_mega", F, 5, F, 40, F, F, T), [Way((12, 0), FUSED)]),  # rects + one triangle
    (("k_mega", F, 5, F, 40, F, T, T), [Way(MESH, FUSED, 0, WAIT0)]),
    (("k_mega", F, 6, F, 1, F, T, F), [Way((13, 0), FUSED)]),
    (("k_mega", F, 6, F, 3, F, T, F), [Way((99, 0), FUSED, 4)]),
    (("k_mega", F, 6, F, 5, F, T, F), [Way((8, 0), FUSED, 4)]),
    (("k_mega", T, 3, T, 63, T, F, T), [Way(general_medium, FUSED)]),
    (("k_mega", T, 4, F, 63, T, F, T), [Way((5, 0), FUSED), Way(medium_and_triangles, FUSED)]),
    # k_mega_r<MINB, PM, WIDE>: the fused kernel with resumable traversal (RTB200_MEGA_WAIT lanes end a traversal round)
    (("k_mega_r", 5, 1, F), [Way((13, 0), FUSED, 0, WAIT16)]),
    (("k_mega_r", 5, 3, F), [Way((99, 0), FUSED, 0, WAIT16)]),
    (("k_mega_r", 7, 40, F), [Way(MESH, FUSED, 2)]),
    (("k_mega_r", 7, 40, T), [Way(MESH, FUSED)]),
    # k_pool<PM, WIDE, MEDIA, GENERAL_MEDIA, XF, P, MINB>: every warp runs a wavefront of its own in shared memory
    (("k_pool", 1, T, F, F, F, 128, 4), [Way((13, 0), POOL)]),
    (("k_pool", 40, T, F, F, F, 128, 4), [Way(MESH, POOL)]),
    (("k_pool", 63, F, F, F, T, 128, 4), [Way((4, 0), POOL), Way(wrapped_spheres, POOL)]),
    (("k_pool", 63, F, T, T, T, 128, 4), [Way((5, 0), POOL)]),
]
# Instances in the build that no scene, knob or flag can make launch_render pick, each with the reason.  None at present.
UNREACHABLE = []


def test_decode_kernel_reads_mangled_and_demangled_names():
    for mangled, demangled in (
            ("_ZN3rtb6k_megaILb0ELi6ELb0ELj1ELb0ELb1ELb0EEEvNS_11DeviceSceneENS_6JobDevENS_6QueuesEPl",
             "void rtb::k_mega<false, 6, false, 1u, false, true, false>(rtb::DeviceScene, rtb::JobDev, rtb::Queues, long*)"),
            ("_ZN3rtb10k_extend_pILb0ELb1ELi4EEEvNS_11DeviceSceneENS_6JobDevENS_9PathStateENS_6QueuesEi",
             "void rtb::k_extend_p<false, true, 4>(rtb::DeviceScene, rtb::JobDev, rtb::PathState, rtb::Queues, int)"),
            ("_ZN3rtb6k_poolILj40ELb1ELb0ELb0ELb0ELi128ELi4EEEvNS_11DeviceSceneENS_6JobDevENS_6QueuesEPl",
             "void rtb::k_pool<40u, true, false, false, false, 128, 4>(rtb::DeviceScene, rtb::JobDev, rtb::Queues, long*)")):
        k = decode_kernel(mangled)
        assert k == decode_kernel(demangled) and cxx(k) == cxx(decode_kernel(demangled))
        assert [type(a) for a in k[1:]] == [type(a) for a in decode_kernel(demangled)[1:]]
    assert decode_kernel("_ZN3rtb6k_megaILb0ELi6ELb0ELj1ELb0ELb1ELb0EEEvNS_11DeviceSceneENS_6JobDevENS_6QueuesEPl") == \
        ("k_mega", False, 6, False, 1, False, True, False)
    assert decode_kernel("k_shade_all(rtb::DeviceScene, rtb::JobDev, rtb::PathState, rtb::Queues, long*, int)") is None
    assert decode_kernel("_ZN3rtb11k_mega_initENS_6QueuesE") is None


def test_table_rows_are_well_formed():
    kernels = [k for k, _ in VARIANTS]
    assert len(set(map(cxx, kernels))) == len(kernels), "two rows claim the same kernel"
    assert not set(map(cxx, kernels)) & set(cxx(k) for k, _ in UNREACHABLE)
    for k, ways in VARIANTS:
        assert k[0] in RENDER_KERNELS and ways, k
        wavefront = k[0] in ("k_extend", "k_extend_p")
        for w in ways:
            # COUNT forces the wavefront; the other flags pick the mode the row's kernel belongs to
            assert (w.flags in (WAVE, COUNT)) == wavefront and (w.flags == POOL) == (k[0] == "k_pool"), (cxx(k), w)
            assert (w.flags == COUNT) == (k[0] != "k_pool" and k[2] is True and wavefront), (cxx(k), w)


@pytest.mark.skipif(not os.path.exists(LOG), reason="needs the library built by csrc/Makefile (build/kernels.ptxas.log)")
def test_every_render_kernel_in_the_build_has_a_row():
    built = {cxx(k) for k in log_instances()}
    claimed = [cxx(k) for k, _ in VARIANTS] + [cxx(k) for k, _ in UNREACHABLE]
    assert len(built) >= len(RENDER_KERNELS)
    assert sorted(built - set(claimed)) == [], "render kernels in the build that no row of VARIANTS claims"
    assert sorted(set(claimed) - built) == [], "rows of VARIANTS for kernels the build does not contain"
    assert len(claimed) == len(set(claimed))


# ---------------------------------------------------------------- GPU helpers
def kernels_run(fn):
    """-> (fn(), {render kernels the CUDA activity trace of fn() recorded})"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
    ran = set()
    for ev in prof.events():
        if ev.device_type.name == "CUDA":
            k = decode_kernel(ev.name)
            if k is not None:
                ran.add(cxx(k))
    return out, ran


def gpu_scene(scene, width=0, env=(), monkeypatch=None):
    for k, v in env:
        monkeypatch.setenv(k, v)
    g = rtb.new_scene()  # rt_scene_create reads the RTB200_* knobs
    for k, _ in env:
        monkeypatch.delenv(k)
    build(scene, g, width)
    return g


_REF, _ORC = {}, {}


def reference(scene, cfg):
    """(accumulator, segments) of a product scene with default knobs, cached per scene and config"""
    key = (scene_name(scene), cfg.image_width, cfg.aspect_ratio, cfg.samples_per_pixel, cfg.seed, cfg.sample_begin, cfg.sample_end, cfg.flags)
    if key not in _REF:
        g = gpu_scene(scene)
        _, acc, st = g.render(cfg, want_accum=True)
        _REF[key] = (acc, st["segments"])
        g.close()
    return _REF[key]


def oracle_render(orc, scene, cfg):
    key = (scene_name(scene), cfg.image_width, cfg.aspect_ratio, cfg.samples_per_pixel, cfg.seed, cfg.sample_begin, cfg.sample_end)
    if key not in _ORC:
        o = orc.new_scene()
        build(scene, o)
        _ORC[key] = o.render(cfg, want_accum=True)
        o.close()
    return _ORC[key]


def assert_e2_bar(sg, ag, stg, so, ao, sto):
    """the sample-by-sample bar of test_E2_render_matches_oracle_sample_by_sample"""
    assert stg["paths"] == sto["paths"]
    fg, fo = ag / capi.ACCUM_SCALE, ao / capi.ACCUM_SCALE
    pix_bad = (np.abs(fg - fo) / np.maximum(1e-3, np.abs(fo)) > 1e-5).any(axis=2)
    assert pix_bad.mean() < 0.02, (pix_bad.mean(), stg, sto)
    assert abs(fg.mean() - fo.mean()) <= 0.01 * max(fo.mean(), 1e-3)
    assert abs(stg["segments"] - sto["segments"]) <= 0.005 * sto["segments"]
    assert (np.abs(sg - so) > 1).any(axis=2).mean() < 0.02


def make_cfg(W, aspect, spp, seed, flags=0, *, sample_begin=0, sample_end=0):
    return capi.make_config(W, aspect, spp, 50, seed=seed, flags=flags, sample_begin=sample_begin, sample_end=sample_end)


# ---------------------------------------------------------------- every row on the GPU
CASES = [pytest.param(k, w, id=f"{cxx(k)}-{scene_name(w.scene)}-f{w.flags}-w{w.width}" + "".join(f"-{n[7:]}{v}" for n, v in w.env))
         for k, ways in VARIANTS for w in ways]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,way", CASES)
def test_variant_runs_its_kernel_and_matches_the_wavefront_and_the_oracle(orc, kernel, way, monkeypatch):
    wavefront = kernel[0] in ("k_extend", "k_extend_p")
    W, aspect, spp, seed = 72, aspect_of(way.scene), 4, 21
    ref_acc, ref_segs = reference(way.scene, make_cfg(W, aspect, spp, seed, FUSED if wavefront else WAVE))
    g = gpu_scene(way.scene, way.width, way.env, monkeypatch)
    cfg = make_cfg(W, aspect, spp, seed, way.flags)
    (sg, ag, stg), ran = kernels_run(lambda: g.render(cfg, want_accum=True))
    assert ran == {cxx(kernel)}, ran
    assert np.array_equal(ag, ref_acc) and stg["segments"] == ref_segs
    assert ag.any()
    if way.flags == COUNT:  # the counting pass renders what the same scene renders without counting
        _, a_plain, st_plain = g.render(make_cfg(W, aspect, spp, seed, WAVE), want_accum=True)
        assert np.array_equal(ag, a_plain) and stg["segments"] == st_plain["segments"]
        assert stg["box_tests"] > 0
    g.close()
    so, ao, sto = oracle_render(orc, way.scene, make_cfg(W, aspect, spp, seed))
    assert_e2_bar(sg, ag, stg, so, ao, sto)


# ---------------------------------------------------------------- edges of the path enumeration, per kernel family
Family = namedtuple("Family", "scene flags width kernel ties")
FAMILIES = {
    "wavefront": Family((13, 0), WAVE, 0, ("k_extend", F, F, 5, F, 63, F), False),
    "fused_pairs": Family((13, 0), FUSED, 2, ("k_mega", F, 5, F, 1, F, F, T), False),
    "wide_sphere_camera_batches": Family((13, 0), FUSED, 0, ("k_mega", F, 6, F, 1, F, T, F), False),
    "resumable_mesh": Family(MESH, FUSED, 0, ("k_mega_r", 7, 40, T), True),  # f32 triangles: documented grazing cases
    "media_fused": Family((5, 0), FUSED, 0, ("k_mega", T, 4, F, 63, T, F, T), False),
    "pool": Family((13, 0), POOL, 0, ("k_pool", 1, T, F, F, F, 128, 4), False),
}


def render_paths(g, cfg, ranges, H):
    """rt_render_device_paths over each [b, e) of `ranges`, summed into one device accumulator -> (accumulator, paths)"""
    import torch
    api = rtb.load()
    acc = torch.zeros((H, cfg.image_width, 3), dtype=torch.int64, device="cuda")
    stream = torch.cuda.current_stream()
    paths = 0
    for b, e in ranges:
        st = capi.Stats()
        api.check(api.render_device_paths(g.h, C.byref(cfg), b, e, C.c_void_p(acc.data_ptr()), C.c_void_p(stream.cuda_stream), C.byref(st)))
        paths += st.paths
    torch.cuda.synchronize()
    return acc.cpu().numpy(), paths


def family_scenes(f):
    """(the family's scene, the same scene with default knobs for the other mode, the flags of that mode)"""
    return gpu_scene(f.scene, f.width), gpu_scene(f.scene), (FUSED if f.flags == WAVE else WAVE)


@pytest.mark.gpu
@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_tails_of_the_path_enumeration(orc, family):
    # renders of 1, 31, 33 and 129 paths (path ranges that start inside a sample) and a whole render of 129 x 127 x 127 = 2 080 641
    # paths, 32 k + 1: the last claimed chunk and the last camera batch hold one path
    f = FAMILIES[family]
    g, gr, rflags = family_scenes(f)
    o = orc.new_scene()
    build(f.scene, o)
    W, aspect, spp = 40, aspect_of(f.scene), 4
    cfg, cfg_r = make_cfg(W, aspect, spp, 31, f.flags), make_cfg(W, aspect, spp, 31, rflags)
    H = g.image_height(cfg)
    npix = W * H
    for n in (1, 31, 33, 129):
        b = npix + 5 + n  # sample 1, from pixel 5 + n on
        acc, paths = render_paths(g, cfg, [(b, b + n)], H)
        acc_r, paths_r = render_paths(gr, cfg_r, [(b, b + n)], H)
        assert paths == paths_r == n and np.array_equal(acc, acc_r), (family, n)
        L = np.arange(b, b + n, dtype=np.uint64)
        pix, smp = L % np.uint64(npix), L // np.uint64(npix)
        assert np.count_nonzero(acc.reshape(-1, 3).any(axis=1)) <= n and not acc.reshape(-1, 3)[np.setdiff1d(np.arange(npix), pix.astype(np.int64))].any()
        if not f.ties:  # every pixel within the E2 per-pixel bar of the oracle's radiance of the same paths
            rad = np.zeros((npix, 3))
            np.add.at(rad, pix.astype(np.int64), orc.path_radiance(o, cfg, pix * np.uint64(spp) + smp))
            fg = acc.reshape(-1, 3) / capi.ACCUM_SCALE
            assert (np.abs(fg - rad) <= 1e-5 * np.maximum(1e-3, np.abs(rad))).all(), (family, n)
    o.close()
    big, big_r = make_cfg(129, 129 / 127.5, 127, 32, f.flags), make_cfg(129, 129 / 127.5, 127, 32, rflags)
    (sg, ag, stg), ran = kernels_run(lambda: g.render(big, want_accum=True))
    _, ar, str_ = gr.render(big_r, want_accum=True)
    assert ran == {cxx(f.kernel)}, ran
    assert stg["paths"] == 129 * 127 * 127 and stg["paths"] % 32 == 1
    assert np.array_equal(ag, ar) and stg["segments"] == str_["segments"]
    if not f.ties:
        assert_e2_bar(sg, ag, stg, *oracle_render(orc, f.scene, make_cfg(129, 129 / 127.5, 127, 32)))
    g.close()
    gr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_path_ids_past_2_32(orc, family):
    # 64 x 40 pixels at 2^21 samples per pixel, samples [2^21 - 3, 2^21): every pixel from 2048 on has path ids past 2^32
    f = FAMILIES[family]
    g, gr, rflags = family_scenes(f)
    spp = 1 << 21
    s0 = spp - 3
    aspect = 64 / 40.5
    sg, ag, stg = g.render(make_cfg(64, aspect, spp, 41, f.flags, sample_begin=s0, sample_end=spp), want_accum=True)
    _, ar, str_ = gr.render(make_cfg(64, aspect, spp, 41, rflags, sample_begin=s0, sample_end=spp), want_accum=True)
    assert ag.shape == (40, 64, 3) and stg["paths"] == 64 * 40 * 3 and 2048 * spp >= 1 << 32
    assert np.array_equal(ag, ar) and stg["segments"] == str_["segments"]
    assert ag[32:].any()  # rows 32.. = pixels 2048..
    assert_e2_bar(sg, ag, stg, *oracle_render(orc, f.scene, make_cfg(64, aspect, spp, 41, sample_begin=s0, sample_end=spp)))
    g.close()
    gr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_enumeration_indices_past_2_32_and_2_33(family):
    # 64 x 40 pixels at 2^22 samples per pixel: 1.07e10 sample-major indices.  Ranges that straddle 2^32 and 2^33, rendered next to
    # their neighbours by rt_render_device_paths, sum to rt_render over the two samples that cover them, bit for bit
    f = FAMILIES[family]
    g = gpu_scene(f.scene, f.width)
    spp, npix = 1 << 22, 64 * 40
    aspect = 64 / 40.5
    cfg = make_cfg(64, aspect, spp, 51, f.flags)
    for X in (1 << 32, 1 << 33):
        sa = X // npix
        lo, hi = sa * npix, (sa + 2) * npix
        assert lo < X - 1 and X + 1 < hi
        acc, paths = render_paths(g, cfg, [(lo, X - 1), (X - 1, X + 1), (X + 1, hi)], 40)
        _, whole, st = g.render(make_cfg(64, aspect, spp, 51, f.flags, sample_begin=sa, sample_end=sa + 2), want_accum=True)
        assert paths == st["paths"] == 2 * npix
        assert np.array_equal(acc, whole) and whole.any(), (family, X)
    g.close()


def miss_everything(s):
    """a constant background and small spheres behind the camera: every path ends at its first segment"""
    m = s.lambertian((0.5, 0.5, 0.5))
    s.set_root(s.list([s.sphere((0.3 * k - 1, 0.2 * (k % 3), 10), 0.1, m) for k in range(8)]))
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 40, 1.0, 0.0, 10, 0, 1)
    s.set_background((0.3, 0.55, 0.8))


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [FUSED, WAVE, POOL], ids=["fused", "wavefront", "pool"])
def test_one_render_of_more_than_2_32_paths(flags):
    # 256 x 256 pixels at 65 537 samples: 4 295 032 832 paths, every one a miss.  Each sample adds floor(bg * 2^32 + 0.5) of the
    # f32 background to its pixel, so every channel of every pixel holds 65 537 times that
    g = gpu_scene(miss_everything)
    (_, _, _), ran = kernels_run(lambda: g.render(make_cfg(64, 1.0, 2, 61, flags), want_accum=True))
    expect = {FUSED: ("k_mega", F, 6, F, 1, F, T, F), WAVE: ("k_extend", F, F, 5, F, 63, F), POOL: ("k_pool", 1, T, F, F, F, 128, 4)}[flags]
    assert ran == {cxx(expect)}, ran
    spp = 65537
    t0 = time.perf_counter()
    _, acc, st = g.render(make_cfg(256, 1.0, spp, 61, flags), want_accum=True)
    wall = time.perf_counter() - t0
    print(f"\n{cxx(expect)}: {st['paths']} paths in {wall:.3f} s ({st['ms_device']:.1f} ms device)")
    g.close()
    n = 256 * 256 * spp
    assert n > 1 << 32 and st["paths"] == st["segments"] == n
    per = np.floor(np.float32([0.3, 0.55, 0.8]).astype(np.float64) * 2.0 ** 32 + 0.5).astype(np.int64) * spp
    assert acc.shape == (256, 256, 3) and (acc == per).all()
