"""Denoised renders (rt_render_aov, rt_render_denoised, ray_tracing_series_rust_b200/denoise.py).

CPU: the oracle's feature sums (orc_render_aov, tests/oracle_aov) against known answers and their sample-range additivity; the numpy
filter on constant images, albedo and normal steps, unrendered rows and a brute-force loop; k_aov's per-path body compiled for the host
(tests/host_emul/emul_aov.cpp) against the oracle; argument checks of both entry points on a scene that was never committed and the
rt_denoise_config layout.
GPU: rt_render_aov against the oracle, additive over sample ranges and independent of the mode flags; rt_render_denoised's accumulator
equal to rt_render's, its outputs identical in every render mode and equal to denoise.py over rt_render sample ranges and rt_render_aov;
the quality bars against independent-seed references."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import ray_tracing_series_rust_b200 as rtb
from ray_tracing_series_rust_b200 import capi, denoise

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))
RT_ERR_INVALID, RT_ERR_STATE = -1, -2
FLAGS = {"wavefront": 4, "fused": 8, "pool": 16, "auto": 0}
SCALE = capi.ACCUM_SCALE
DEFAULTS = dict(iterations=5, sigma_color=4.0, sigma_albedo=0.1, sigma_normal=0.125)


# ---------------------------------------------------------------- test libraries: the oracle with orc_render_aov, the host emulation


@pytest.fixture(scope="module")
def orc_aov(tmp_path_factory):
    """The oracle (oracle_capi.cpp as it is) plus orc_render_aov, built fresh with oracle/Makefile's flags."""
    so = str(tmp_path_factory.mktemp("orc_aov") / "liboracle_aov.so")
    subprocess.check_call(["g++", "-O3", "-march=x86-64-v3", "-ffp-contract=off", "-std=c++17", "-fPIC", "-fvisibility=hidden", "-pthread",
                           "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "ray_tracing_series_rust_b200", "csrc", "host"),
                           "-shared", "-o", so, os.path.join(HERE, "oracle_aov", "oracle_aov.cpp")])
    return capi.Api(C.CDLL(so), "orc_")


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emul_aov") / "libemul_aov.so")
    cuda_include = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-Wno-unknown-pragmas", "-I" + cuda_include,
                           os.path.join(HERE, "host_emul", "emul_aov.cpp"), "-o", so])
    lib = C.CDLL(so)
    lib.emul_aov_sizeof_device_scene.restype = C.c_uint64
    lib.emul_render_aov.restype = C.c_int32
    lib.emul_render_aov.argtypes = [C.c_void_p] + [C.c_int32] * 6 + [C.c_uint64, C.c_int32, C.c_void_p, C.c_void_p]
    if not os.path.exists(rtb.LIB_PATH):
        rtb.build()
    return lib


def orc_world(api, scene_id, seed=3, param=0):
    o = capi.Scene(api)
    o.world_build(scene_id, seed, param)
    o.commit()
    return o


def aov_mismatch(g, o):
    """fraction of pixels whose albedo or normal sums differ by more than 1e-5 relative (floor 1e-3 per sample mean)"""
    bad = np.zeros(g[0].shape[:2], dtype=bool)
    for x, y in zip(g, o):
        bad |= (np.abs(x - y) > 1e-5 * np.maximum(1e-3 * SCALE, np.abs(y))).any(axis=2)
    return bad.mean()


# ---------------------------------------------------------------- oracle known answers


def one_sphere(api, kind, background=(0.2, 0.4, 0.6)):
    """a unit sphere at the origin seen head-on from z = 5 (aperture 0), material `kind`"""
    s = capi.Scene(api)
    if kind == "lambertian":
        m = s.lambertian((0.3, 0.5, 0.7))
    elif kind == "dielectric":
        m = s.dielectric(1.5)
    elif kind == "light":
        m = s.diffuse_light((4.0, 0.5, 2.0))
    elif kind == "metal":
        m = s.metal((0.8, 0.6, 0.2), 0.3)
    if kind == "medium":
        b = s.sphere((0, 0, 0), 1.0, s.lambertian((0.5, 0.5, 0.5)))
        root = s.constant_medium((0.25, 0.5, 0.75), 1e6, b)
    else:
        root = s.sphere((0, 0, 0), 1.0, m)
    s.set_root(s.list([root]))
    s.set_camera((0, 0, 5), (0, 0, 0), (0, 1, 0), 40.0, 1.0, 0.0, 5.0, 0.0, 1.0)
    s.set_background(background)
    s.commit()
    return s


def fx(x):
    return int(np.rint(x * SCALE))


@pytest.mark.parametrize("kind,albedo", [("lambertian", (0.3, 0.5, 0.7)), ("dielectric", (1, 1, 1)), ("light", (1.0, 0.5, 1.0)),
                                         ("metal", (0.8, 0.6, 0.2)), ("medium", (0.25, 0.5, 0.75))])
def test_oracle_aov_known_answers(orc_aov, kind, albedo):
    s = one_sphere(orc_aov, kind)
    m = 6
    cfg = capi.make_config(41, 1.0, m, 10, seed=5)
    a, n, st = s.render_aov(cfg, raw=True)
    assert st["paths"] == st["segments"] == 41 * 41 * m
    want = [m * fx(x) for x in albedo]
    assert list(a[20, 20]) == want, (a[20, 20], want)         # the centre pixel sees the sphere
    assert list(a[0, 0]) == [m * fx(x) for x in (0.2, 0.4, 0.6)] and (n[0, 0] == 0).all()  # a corner misses: the background
    nm = n[20, 20] / SCALE / m
    if kind == "medium":
        assert (n[20, 20] == 0).all()
    else:
        assert nm[2] > 0.99 and abs(nm[0]) < 0.1 and abs(nm[1]) < 0.1, nm  # faces the camera


def test_oracle_aov_miss_clamps_the_background(orc_aov):
    s = one_sphere(orc_aov, "lambertian", background=(1.7, -0.2, 0.5))
    a, n, _ = s.render_aov(capi.make_config(9, 1.0, 3, 10, seed=1), raw=True)
    assert list(a[0, 0]) == [3 * fx(1.0), 0, 3 * fx(0.5)]


def test_oracle_aov_sample_ranges_add_up(orc_aov):
    o = orc_world(orc_aov, 4)
    full = o.render_aov(capi.make_config(24, 1.0, 7, 10, seed=2, sample_end=5), raw=True)
    p1 = o.render_aov(capi.make_config(24, 1.0, 7, 10, seed=2, sample_end=2), raw=True)
    p2 = o.render_aov(capi.make_config(24, 1.0, 7, 10, seed=2, sample_begin=2, sample_end=5), raw=True)
    assert np.array_equal(p1[0] + p2[0], full[0]) and np.array_equal(p1[1] + p2[1], full[1])


# ---------------------------------------------------------------- the numpy filter


def _inputs(H, W, c, albedo, normal, n=8, rows=None, rng=None, noise=0.0):
    """A = B = c with optional noise, features constant per pixel as given (arrays or triples)"""
    hA, hB = denoise.split(n)
    base = np.broadcast_to(np.asarray(c, dtype=np.float64), (H, W, 3))
    ea = base if rng is None else base + noise * rng.standard_normal((H, W, 3))
    eb = base if rng is None else base + noise * rng.standard_normal((H, W, 3))
    A = np.rint(ea * hA * SCALE).astype(np.int64)
    B = np.rint(eb * hB * SCALE).astype(np.int64)
    m = 4
    al = np.rint(np.broadcast_to(np.asarray(albedo, dtype=np.float64), (H, W, 3)) * SCALE).astype(np.int64) * m
    nm = np.rint(np.broadcast_to(np.asarray(normal, dtype=np.float64), (H, W, 3)) * SCALE).astype(np.int64) * m
    return A, B, hA, hB, al, nm, m


def test_constant_image_is_unchanged():
    H, W = 11, 13
    A, B, hA, hB, al, nm, m = _inputs(H, W, (0.3, 0.6, 0.9), (0.5, 0.5, 0.5), (0, 0, 1))
    out = denoise.denoise(A, B, hA, hB, al, nm, m, H, 5, **{k: v for k, v in DEFAULTS.items() if k != "iterations"})
    c, _, _, _ = denoise.filter_inputs(A, B, hA, hB, al, nm, m, H)
    assert np.allclose(out, c, rtol=1e-14, atol=0)


def _step_weight(feature):
    """the weight across a feature step at the default sigmas, relative to the centre tap's, for a noise-free colour"""
    H, W = 6, 8
    al = np.full((H, W, 3), 0.5)
    nm = np.zeros((H, W, 3))
    nm[..., 2] = 1.0
    if feature == "albedo":
        al[:, 4:] = 1.0  # a step of 0.5
    else:
        nm[:, 4:] = (1.0, 0.0, 0.0)  # 90 degrees
    A, B, hA, hB, alS, nmS, m = _inputs(H, W, (0.4, 0.4, 0.4), al, nm)
    c, v, a, n = denoise.filter_inputs(A, B, hA, hB, alS, nmS, m, H)
    da = ((a[:, 3] - a[:, 4]) ** 2).sum(axis=-1) / DEFAULTS["sigma_albedo"] ** 2
    dn = ((n[:, 3] - n[:, 4]) ** 2).sum(axis=-1) / DEFAULTS["sigma_normal"] ** 2
    return float(np.exp(-(da + dn)).max()), (A, B, hA, hB, alS, nmS, m, H, W)


@pytest.mark.parametrize("feature", ["albedo", "normal"])
def test_feature_steps_are_not_blurred(feature):
    w, (A, B, hA, hB, alS, nmS, m, H, W) = _step_weight(feature)
    assert w < 1e-6
    # a colour step on the same edge survives five passes: the two sides keep their own values
    A2, B2 = A.copy(), B.copy()
    A2[:, 4:] *= 2
    B2[:, 4:] *= 2
    out = denoise.denoise(A2, B2, hA, hB, alS, nmS, m, H, 5, **{k: v for k, v in DEFAULTS.items() if k != "iterations"})
    c, _, _, _ = denoise.filter_inputs(A2, B2, hA, hB, alS, nmS, m, H)
    assert np.allclose(out, c, rtol=1e-6, atol=0)


def test_unrendered_rows_stay_zero_and_are_never_read():
    H, W, rows = 9, 10, 6
    rng = np.random.default_rng(1)
    A, B, hA, hB, al, nm, m = _inputs(H, W, (0.3, 0.2, 0.1), (0.5, 0.5, 0.5), (0, 0, 1), rng=rng, noise=0.05)
    ref = denoise.denoise(A, B, hA, hB, al, nm, m, rows, 3, 4.0, 0.1, 0.125)
    junk = [x.copy() for x in (A, B, al, nm)]
    for x in junk:
        x[rows:] = 123456789
    out = denoise.denoise(junk[0], junk[1], hA, hB, junk[2], junk[3], m, rows, 3, 4.0, 0.1, 0.125)
    assert (out[rows:] == 0).all()
    assert np.array_equal(out, ref)


def test_one_iteration_equals_a_brute_force_loop():
    H = W = 7
    rng = np.random.default_rng(7)
    n = 9
    hA, hB = denoise.split(n)
    A = rng.integers(0, 3 << 32, size=(H, W, 3), dtype=np.int64)
    B = rng.integers(0, 3 << 32, size=(H, W, 3), dtype=np.int64)
    m = 3
    al = rng.integers(0, m << 32, size=(H, W, 3), dtype=np.int64)
    nm = rng.integers(-(m << 32), m << 32, size=(H, W, 3), dtype=np.int64)
    sc, sa, sn = 2.0, 0.3, 0.5
    got = denoise.denoise(A, B, hA, hB, al, nm, m, H, 1, sc, sa, sn)
    # written out independently, pixel by pixel
    S = 2.0 ** -32
    L = lambda x: 0.2126 * x[0] + 0.7152 * x[1] + 0.0722 * x[2]
    c = (A + B) * S / n
    v = (L((A * S / hA).transpose(2, 0, 1)) - L((B * S / hB).transpose(2, 0, 1))) ** 2 * hA * hB / n ** 2
    fa, fn = al * S / m, nm * S / m
    g, h = [0.25, 0.5, 0.25], [1 / 16, 1 / 4, 3 / 8, 1 / 4, 1 / 16]
    want = np.zeros_like(got)
    for y in range(H):
        for x in range(W):
            num = den = 0.0
            for yy in range(max(0, y - 1), min(H, y + 2)):
                for xx in range(max(0, x - 1), min(W, x + 2)):
                    num += g[yy - y + 1] * g[xx - x + 1] * v[yy, xx]
                    den += g[yy - y + 1] * g[xx - x + 1]
            vb = num / den
            ws, acc = 0.0, np.zeros(3)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    qy, qx = y + dy, x + dx
                    if not (0 <= qy < H and 0 <= qx < W):
                        continue
                    e = abs(L(c[y, x]) - L(c[qy, qx])) / (sc * np.sqrt(vb) + 1e-10)
                    e += ((fa[y, x] - fa[qy, qx]) ** 2).sum() / sa ** 2 + ((fn[y, x] - fn[qy, qx]) ** 2).sum() / sn ** 2
                    w = h[dx + 2] * h[dy + 2] * np.exp(-e)
                    ws += w
                    acc += w * c[qy, qx]
            want[y, x] = acc / ws
    assert np.allclose(got, want, rtol=1e-12, atol=1e-15)


def test_screen_values_quantise_like_rt_render():
    x = np.array([0.0, 0.25, 1.0, 4.0, -1.0, np.nan])
    assert list(denoise.screen_values(x)) == [0.0, 127.0, 255.0, 255.0, 0.0, 0.0]


# ---------------------------------------------------------------- host emulation of k_aov's body against the oracle


@pytest.mark.parametrize("scene_id,aspect", [(4, 1.0), (5, 1.0), (6, 1.0), (13, 1.5)])
def test_host_emulated_aov_matches_oracle(emul, orc_aov, scene_id, aspect):
    W, spp, s0, s1, seed = 24, 6, 1, 4, 9
    g = rtb.new_scene()
    g.world_build(scene_id, 3, 0)
    ds = g.debug_host_scene(emul.emul_aov_sizeof_device_scene())
    cfg = capi.make_config(W, aspect, spp, 10, seed=seed, sample_begin=s0, sample_end=s1)
    H = g.image_height(cfg)
    o = orc_world(orc_aov, scene_id)
    oa, on, _ = o.render_aov(cfg, raw=True)
    ga, gn = np.zeros((H, W, 3), np.int64), np.zeros((H, W, 3), np.int64)
    for wd in (0, 1) if scene_id == 13 else (0,):  # scene 13 carries the 4-wide tree k_aov<true> walks
        ga[:] = 0
        gn[:] = 0
        assert emul.emul_render_aov(ds, W, H, H, spp, s0, s1, seed, wd, ga.ctypes.data, gn.ctypes.data) == 0
        assert aov_mismatch((ga, gn), (oa, on)) < 0.03, wd
    g.close()


# ---------------------------------------------------------------- argument checks (no GPU)


@pytest.fixture(scope="module")
def api():
    if not os.path.exists(rtb.LIB_PATH):
        rtb.build()
    api = rtb.load()
    api.lib.rt_render_denoised.restype, api.lib.rt_render_denoised.argtypes = capi.RENDER_DENOISED_SIGNATURE
    api.lib.rt_render_aov.restype, api.lib.rt_render_aov.argtypes = capi.RENDER_AOV_SIGNATURE
    return api


def test_denoise_config_layout():
    assert C.sizeof(capi.DenoiseConfig) == 32
    assert capi.DenoiseConfig.sigma_color.offset == 8 and capi.DenoiseConfig.sigma_normal.offset == 24


def test_render_denoised_argument_checks(api):
    s = rtb.new_scene()  # never committed: every rejection below comes from the argument checks
    cfg = capi.make_config(32, 1.0, 16, 5)

    def dc(**kw):
        d = dict(aov_samples=4, **DEFAULTS)
        d.update(kw)
        return capi.DenoiseConfig(d["aov_samples"], d["iterations"], d["sigma_color"], d["sigma_albedo"], d["sigma_normal"])

    def call(c, d):
        return api.lib.rt_render_denoised(s.h, C.byref(c), C.byref(d) if d is not None else None, None, None, None, None)

    bad = [None, dc(aov_samples=0), dc(aov_samples=17), dc(iterations=0), dc(iterations=9)]
    for k in ("sigma_color", "sigma_albedo", "sigma_normal"):
        bad += [dc(**{k: 0.0}), dc(**{k: -1.0}), dc(**{k: float("nan")}), dc(**{k: float("inf")})]
    for d in bad:
        assert call(cfg, d) == RT_ERR_INVALID
    for c in (capi.make_config(32, 1.0, 1, 5), capi.make_config(32, 1.0, 16, 5, flags=(1 << 16) | (2 << 24)), capi.make_config(32, 1.0, 16, 5, flags=32),
              capi.make_config(32, 1.0, 16, 5, sample_begin=1), capi.make_config(32, 1.0, 16, 5, sample_end=8)):
        assert call(c, dc(aov_samples=1)) == RT_ERR_INVALID
    assert api.lib.rt_render_denoised(None, C.byref(cfg), C.byref(dc()), None, None, None, None) == RT_ERR_INVALID
    assert api.lib.rt_render_denoised(s.h, None, C.byref(dc()), None, None, None, None) == RT_ERR_INVALID
    for c, d in ((cfg, dc()), (cfg, dc(aov_samples=16, iterations=8)), (capi.make_config(32, 1.0, 2, 5, sample_end=2, flags=8), dc(aov_samples=1, iterations=1)),
                 (capi.make_config(32, 1.0, 16, 5, flags=1 << 24), dc())):
        assert call(c, d) == RT_ERR_STATE
    # rt_render_aov: tile shards and no-wait are refused, the rest needs a committed scene
    for flags in ((1 << 16) | (2 << 24), 32):
        assert api.lib.rt_render_aov(s.h, C.byref(capi.make_config(32, 1.0, 16, 5, flags=flags)), None, None, None) == RT_ERR_INVALID
    assert api.lib.rt_render_aov(s.h, None, None, None, None) == RT_ERR_INVALID
    assert api.lib.rt_render_aov(s.h, C.byref(capi.make_config(32, 1.0, 16, 5, flags=4)), None, None, None) == RT_ERR_STATE
    s.close()


# ---------------------------------------------------------------- GPU


def _gpu_scene(scene_id, param=0, seed=3):
    g = rtb.new_scene()
    g.world_build(scene_id, seed, param)
    g.commit()
    return g


AOV_SCENES = [(4, 0, 1.0), (5, 0, 1.0), (6, 0, 1.0), (8, 0, 1.0), (13, 0, 1.5), (99, 0, 16 / 9), (14, 48, 1.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,param,aspect", AOV_SCENES)
def test_gpu_aov_matches_oracle(orc_aov, scene_id, param, aspect):
    g = _gpu_scene(scene_id, param)
    o = orc_world(orc_aov, scene_id, param=param)
    cfg = capi.make_config(40, aspect, 8, 10, seed=11, sample_begin=2, sample_end=6)
    ga, gn, st = g.render_aov(cfg, raw=True)
    oa, on, _ = o.render_aov(cfg, raw=True)
    H = g.image_height(cfg)
    assert st["paths"] == st["segments"] == 40 * H * 4
    bad = aov_mismatch((ga, gn), (oa, on))
    assert bad < 0.03, f"feature sums differ from the oracle on {bad:.2%} of the pixels"
    # sample ranges add up bit for bit, and no mode flag changes the result
    p1 = g.render_aov(capi.make_config(40, aspect, 8, 10, seed=11, sample_begin=2, sample_end=3), raw=True)
    p2 = g.render_aov(capi.make_config(40, aspect, 8, 10, seed=11, sample_begin=3, sample_end=6), raw=True)
    assert np.array_equal(p1[0] + p2[0], ga) and np.array_equal(p1[1] + p2[1], gn)
    for flags in FLAGS.values():
        fa, fn, _ = g.render_aov(capi.make_config(40, aspect, 8, 10, seed=11, sample_begin=2, sample_end=6, flags=flags), raw=True)
        assert np.array_equal(fa, ga) and np.array_equal(fn, gn), flags
    g.close()


DENOISE_CASES = [  # scene, param, aspect, W, spp, aov_samples, iterations, compat_threads
    (13, 0, 1.5, 64, 16, 8, 5, 0),
    (4, 0, 1.0, 48, 9, 3, 1, 0),      # odd spp: hA = 4, hB = 5
    (6, 0, 1.0, 48, 12, 12, 8, 0),
    (5, 0, 1.0, 40, 7, 2, 3, 0),
    (14, 48, 1.0, 40, 6, 6, 4, 0),
    (13, 0, 1.5, 64, 10, 4, 5, 5),    # compat_threads = 5: 42 = 8 * 5 + 2 rows, the top two unrendered
]


def _reference(g, W, aspect, spp, m, its, compat, seed, sigmas):
    hA, hB = denoise.split(spp)
    A = g.render(capi.make_config(W, aspect, spp, 50, seed=seed, compat_threads=compat, sample_end=hA), want_accum=True)[1]
    B = g.render(capi.make_config(W, aspect, spp, 50, seed=seed, compat_threads=compat, sample_begin=hA), want_accum=True)[1]
    al, nm, _ = g.render_aov(capi.make_config(W, aspect, spp, 50, seed=seed, compat_threads=compat, sample_end=m), raw=True)
    H = A.shape[0]
    rows = (H // compat) * compat if compat else H
    lin = denoise.denoise(A, B, hA, hB, al, nm, m, rows, its, *sigmas)
    return A + B, lin, rows


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,param,aspect,W,spp,m,its,compat", DENOISE_CASES)
def test_denoised_equals_numpy_reference(scene_id, param, aspect, W, spp, m, its, compat):
    g = _gpu_scene(scene_id, param)
    sig = (4.0, 0.1, 0.125)
    acc_ref, lin_ref, rows = _reference(g, W, aspect, spp, m, its, compat, 6, sig)
    full = g.render(capi.make_config(W, aspect, spp, 50, seed=6, compat_threads=compat), want_accum=True)[1]
    assert np.array_equal(acc_ref, full)
    first = None
    for mode, flags in FLAGS.items():
        cfg = capi.make_config(W, aspect, spp, 50, seed=6, compat_threads=compat, flags=flags)
        screen, lin, acc, st = g.render_denoised(cfg, aov_samples=m, iterations=its, sigma_color=sig[0], sigma_albedo=sig[1], sigma_normal=sig[2])
        assert np.array_equal(acc, full), mode
        assert st["paths"] == W * rows * spp, mode
        if first is None:
            first = (screen, lin)
            assert (lin[rows:] == 0).all() and (screen[rows:] == 0).all()
            assert np.allclose(lin, lin_ref, rtol=1e-9, atol=1e-300), np.abs(lin - lin_ref).max()
            ref_screen = denoise.screen_values(lin_ref, rows)
            q = 255.9 * np.sqrt(np.clip(lin_ref, 0, None))
            tie = np.abs(q - np.rint(q)) < 1e-9 * np.maximum(1.0, q)
            assert ((screen == ref_screen) | tie).all()
        else:
            assert np.array_equal(screen, first[0]) and np.array_equal(lin, first[1]), mode
    g.close()


def _rmse(x, ref):
    return float(np.sqrt(np.mean((x - ref) ** 2)))


QUALITY = [  # scene, param, aspect, W, spp, reference spp, bar (denoised RMSE / raw RMSE)
    (13, 0, 1.5, 400, 16, 1024, 0.7),
    (4, 0, 1.0, 300, 16, 1024, 0.7),
    (14, 48, 1.0, 256, 16, 1024, 0.7),
    (5, 0, 1.0, 200, 16, 1024, 1.0),
    (6, 0, 1.0, 200, 16, 1024, 1.0),
    # converged: the filter should do no harm.  It does: 1.50 at the defaults, 1.08 at best over the sweep of DESIGN.md section 11 (the
    # colour stop scales with the noise estimate, so at convergence it passes differences the first-hit features cannot see)
    pytest.param(13, 0, 1.5, 200, 1024, 8192, 1.0, marks=pytest.mark.xfail(strict=True, reason="measured ratio 1.50 at 1024 spp, DESIGN.md section 11")),
]


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,param,aspect,W,spp,ref_spp,bar", QUALITY)
def test_denoised_quality(scene_id, param, aspect, W, spp, ref_spp, bar):
    g = _gpu_scene(scene_id, param)
    ref = g.render(capi.make_config(W, aspect, ref_spp, 50, seed=1000 + scene_id), want_accum=True)[1] / SCALE / ref_spp
    _, lin, acc, _ = g.render_denoised(capi.make_config(W, aspect, spp, 50, seed=7))
    raw = _rmse(acc / SCALE / spp, ref)
    den = _rmse(lin, ref)
    print(f"scene {scene_id} W {W} spp {spp}: raw RMSE {raw:.5f}, denoised {den:.5f}, ratio {den / raw:.3f}")
    assert den <= bar * raw, (den, raw, den / raw)
    g.close()
