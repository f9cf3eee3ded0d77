"""ctypes binding of include/rtb200.h.

One signature table, bound twice: prefix ``rt_`` on librtb200.so (the product) and prefix
``orc_`` on oracle/liboracle_rt.so (the checker, bound from oracle/oracle.py — this module never
loads the oracle).  `Scene` mirrors the C-ABI one method per entry point so that parity tests read
like the reference's scene code (src/world.rs).
"""
from __future__ import annotations

import ctypes as C
import numpy as np

c_d3 = C.POINTER(C.c_double)
c_i32p = C.POINTER(C.c_int32)


class RenderConfig(C.Structure):
    """rt_render_config  [ref: Config, src/world.rs:20-50]"""
    _fields_ = [
        ("image_width", C.c_int32),
        ("aspect_ratio", C.c_double),
        ("samples_per_pixel", C.c_int32),
        ("max_depth", C.c_int32),
        ("compat_threads", C.c_int32),
        ("seed", C.c_uint64),
        ("sample_begin", C.c_int32),
        ("sample_end", C.c_int32),
        ("threads", C.c_int32),
        ("flags", C.c_int32),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("paths", C.c_uint64),
        ("segments", C.c_uint64),
        ("box_tests", C.c_uint64),
        ("prim_tests", C.c_uint64 * 8),
        ("scatters", C.c_uint64 * 5),
        ("medium_queries", C.c_uint64),
        ("iterations", C.c_uint64),
        ("kernel_launches", C.c_uint64),
        ("ms_total", C.c_double),
        ("ms_device", C.c_double),
        ("ms_extend", C.c_double),
    ]

    def as_dict(self):
        return {
            "paths": int(self.paths), "segments": int(self.segments), "box_tests": int(self.box_tests),
            "prim_tests": [int(x) for x in self.prim_tests], "scatters": [int(x) for x in self.scatters],
            "medium_queries": int(self.medium_queries), "iterations": int(self.iterations),
            "kernel_launches": int(self.kernel_launches), "ms_total": float(self.ms_total),
            "ms_device": float(self.ms_device), "ms_extend": float(self.ms_extend),
        }


class AdaptiveConfig(C.Structure):
    """rt_adaptive_config (rt_render_adaptive)"""
    _fields_ = [
        ("min_samples", C.c_int32),
        ("step", C.c_int32),
        ("threshold", C.c_double),
        ("radius", C.c_int32),
    ]


RAY_DTYPE = np.dtype([("o", "<f8", 3), ("d", "<f8", 3), ("time", "<f8")], align=True)
HIT_DTYPE = np.dtype(
    [("prim_id", "<i4"), ("mat_id", "<i4"), ("t", "<f8"), ("p", "<f8", 3), ("normal", "<f8", 3),
     ("u", "<f8"), ("v", "<f8"), ("front_face", "<i4"), ("pad_", "<i4")], align=True)
assert RAY_DTYPE.itemsize == 56 and HIT_DTYPE.itemsize == 88

RT_TRACE_SKIP_MEDIA = 0
RT_TRACE_SEEDED_MEDIA = 1
ACCUM_SCALE = float(2 ** 32)

# name -> (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "scene_create": (_P, []),
    "scene_destroy": (None, [_P]),
    "last_error": (C.c_char_p, []),
    "version": (C.c_char_p, []),
    "tex_solid": (C.c_int32, [_P, c_d3]),
    "tex_checker": (C.c_int32, [_P, C.c_int32, C.c_int32]),
    "tex_noise": (C.c_int32, [_P, C.c_double, c_d3, c_i32p, c_i32p, c_i32p, C.c_uint64]),
    "tex_image": (C.c_int32, [_P, C.c_int32, C.c_int32, c_d3]),
    "tex_image_ppm": (C.c_int32, [_P, C.c_char_p]),
    "mat_lambertian": (C.c_int32, [_P, C.c_int32]),
    "mat_metal": (C.c_int32, [_P, c_d3, C.c_double]),
    "mat_dielectric": (C.c_int32, [_P, C.c_double]),
    "mat_diffuse_light": (C.c_int32, [_P, C.c_int32]),
    "mat_isotropic": (C.c_int32, [_P, C.c_int32]),
    "sphere": (C.c_int32, [_P, c_d3, C.c_double, C.c_int32]),
    "moving_sphere": (C.c_int32, [_P, c_d3, c_d3, C.c_double, C.c_double, C.c_double, C.c_int32]),
    "gravity_sphere": (C.c_int32, [_P, c_d3, C.c_double, C.c_double, C.c_int32]),
    "xy_rect": (C.c_int32, [_P] + [C.c_double] * 5 + [C.c_int32]),
    "xz_rect": (C.c_int32, [_P] + [C.c_double] * 5 + [C.c_int32]),
    "yz_rect": (C.c_int32, [_P] + [C.c_double] * 5 + [C.c_int32]),
    "box": (C.c_int32, [_P, c_d3, c_d3, C.c_int32]),
    "triangle": (C.c_int32, [_P, c_d3, c_d3, c_d3, C.c_int32]),
    "triangle_mesh": (C.c_int32, [_P, c_d3, C.c_int64, C.POINTER(C.c_uint32), C.c_int64, C.c_int32]),
    "ply_load": (C.c_int32, [_P, C.c_char_p, C.c_double, C.c_int32]),
    "list": (C.c_int32, [_P, c_i32p, C.c_int32]),
    "bvh": (C.c_int32, [_P, c_i32p, C.c_int32, C.c_double, C.c_double]),
    "translate": (C.c_int32, [_P, c_d3, C.c_int32]),
    "rotate_y": (C.c_int32, [_P, C.c_double, C.c_int32]),
    "constant_medium": (C.c_int32, [_P, c_d3, C.c_double, C.c_int32]),
    "scene_set_root": (C.c_int32, [_P, C.c_int32]),
    "scene_set_camera": (C.c_int32, [_P, c_d3, c_d3, c_d3] + [C.c_double] * 6),
    "scene_set_camera_fields": (C.c_int32, [_P, c_d3]),
    "scene_set_background": (C.c_int32, [_P, c_d3]),
    "scene_set_background_gradient": (C.c_int32, [_P, c_d3, c_d3]),
    "scene_commit": (C.c_int32, [_P]),
    "world_build": (C.c_int32, [_P, C.c_int32, C.c_uint64, C.c_int32]),
    "scene_num_prims": (C.c_int32, [_P]),
    "render": (C.c_int32, [_P, C.POINTER(RenderConfig), c_d3, C.POINTER(C.c_int64), C.POINTER(Stats)]),
    "image_height": (C.c_int32, [C.POINTER(RenderConfig)]),
    "write_ppm": (C.c_int32, [C.c_char_p, c_d3, C.c_int32, C.c_int32]),
    "render_scene_with_time": (C.c_int32, [_P, C.c_double, C.c_double, C.c_char_p, C.POINTER(RenderConfig), c_d3, C.POINTER(Stats)]),
    "trace_batch": (C.c_int32, [_P, _P, C.c_int64, C.c_double, C.c_double, C.c_int32, C.c_uint64, _P]),
}
# product-only entry points (device-resident accumulators for the multi-GPU path)
DEVICE_SIGNATURES = {
    "render_device": (C.c_int32, [_P, C.POINTER(RenderConfig), _P, _P, C.POINTER(Stats)]),
    "resolve_device": (C.c_int32, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "render_device_paths": (C.c_int32, [_P, C.POINTER(RenderConfig), C.c_uint64, C.c_uint64, _P, _P, C.POINTER(Stats)]),
    # one process, N GPUs: shards rendered per device, accumulators summed + resolved over NVLink peer memory
    "render_multi": (C.c_int32, [_P, C.POINTER(RenderConfig), C.c_int32, C.c_int32, c_d3, C.POINTER(C.c_int64), C.POINTER(Stats)]),
    "scene_commit_multi": (C.c_int32, [_P, C.c_int32]),
    # peer group: the one-process-per-GPU exchange over CUDA IPC + NVLink peer memory (no collective on the data path)
    "peer_create": (_P, [C.c_int32, C.c_int32, C.c_int64, C.POINTER(C.c_uint8)]),
    "peer_connect": (C.c_int32, [_P, C.POINTER(C.c_uint8)]),
    "peer_accum": (_P, [_P]),
    "peer_begin": (C.c_int32, [_P, _P]),
    "peer_publish": (C.c_int32, [_P, _P]),
    "peer_gather_resolve": (C.c_int32, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "peer_timed_out": (C.c_int32, [_P]),
    "peer_destroy": (None, [_P]),
}
# rt_render_adaptive and rt_render_adaptive_multi, bound on first use (Scene.render_adaptive) like the other product-only controls, so that tools can still load
# builds of the library that predate it side by side (tools/ab_multi.py)
RENDER_ADAPTIVE_SIGNATURE = (C.c_int32, [_P, C.POINTER(RenderConfig), C.POINTER(AdaptiveConfig), c_d3, C.POINTER(C.c_int64), c_i32p, C.POINTER(Stats)])
RENDER_ADAPTIVE_MULTI_SIGNATURE = (C.c_int32, [_P, C.POINTER(RenderConfig), C.POINTER(AdaptiveConfig), C.c_int32, c_d3, C.POINTER(C.c_int64), c_i32p,
                                                C.POINTER(Stats)])
RT_PEER_HANDLE_BYTES = 64
RT_SHARD_SAMPLES = 0
RT_SHARD_TILES = 1


class RtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"rt_status {code}: {msg}")
        self.code = code


class Api:
    """The bound function table of one shared library."""

    def __init__(self, lib: C.CDLL, prefix: str, extra=None):
        self.lib = lib
        self.prefix = prefix
        table = dict(SIGNATURES)
        if extra:
            table.update(extra)
        for name, (res, args) in table.items():
            fn = getattr(lib, prefix + name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
            setattr(self, name, fn)

    def err(self) -> str:
        return (self.last_error() or b"").decode("utf-8", "replace")

    def check(self, code: int) -> int:
        if code < 0:
            raise RtError(code, self.err())
        return code


def _d3(v):
    a = (C.c_double * 3)(float(v[0]), float(v[1]), float(v[2]))
    return a


def make_config(image_width, aspect_ratio, samples_per_pixel, max_depth, seed=1, compat_threads=0,
                sample_begin=0, sample_end=0, threads=0, flags=0) -> RenderConfig:
    """Config::new(aspect_ratio, image_width, samples_per_pixel, max_depth, threads)  [ref: world.rs:29-35]"""
    return RenderConfig(int(image_width), float(aspect_ratio), int(samples_per_pixel), int(max_depth),
                        int(compat_threads), int(seed), int(sample_begin), int(sample_end), int(threads), int(flags))


class Scene:
    """One rt_scene* (or the oracle's).  Methods return ids; errors raise RtError."""

    def __init__(self, api: Api):
        self.api = api
        self.h = api.scene_create()
        if not self.h:
            raise RtError(-1, "scene_create failed")

    def close(self):
        if self.h:
            self.api.scene_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _c(self, code):
        return self.api.check(code)

    # ---- textures
    def tex_solid(self, rgb):
        return self._c(self.api.tex_solid(self.h, _d3(rgb)))

    def tex_checker(self, even, odd):
        return self._c(self.api.tex_checker(self.h, even, odd))

    def tex_noise(self, scale, tables=None, seed=0):
        if tables is None:
            return self._c(self.api.tex_noise(self.h, float(scale), None, None, None, None, int(seed)))
        ranvec, px, py, pz = tables
        rv = np.ascontiguousarray(ranvec, dtype=np.float64).reshape(-1)
        ps = [np.ascontiguousarray(p, dtype=np.int32) for p in (px, py, pz)]
        return self._c(self.api.tex_noise(self.h, float(scale), rv.ctypes.data_as(c_d3),
                                          ps[0].ctypes.data_as(c_i32p), ps[1].ctypes.data_as(c_i32p),
                                          ps[2].ctypes.data_as(c_i32p), 0))

    def tex_image(self, texels):
        t = np.ascontiguousarray(texels, dtype=np.float64)
        h, w = t.shape[0], t.shape[1]
        return self._c(self.api.tex_image(self.h, w, h, t.ctypes.data_as(c_d3)))

    def tex_image_ppm(self, path):
        return self._c(self.api.tex_image_ppm(self.h, str(path).encode()))

    # ---- materials
    def lambertian(self, rgb_or_tex):
        tex = rgb_or_tex if isinstance(rgb_or_tex, int) else self.tex_solid(rgb_or_tex)
        return self._c(self.api.mat_lambertian(self.h, tex))

    def metal(self, rgb, fuzz):
        return self._c(self.api.mat_metal(self.h, _d3(rgb), float(fuzz)))

    def dielectric(self, ir):
        return self._c(self.api.mat_dielectric(self.h, float(ir)))

    def diffuse_light(self, rgb_or_tex):
        tex = rgb_or_tex if isinstance(rgb_or_tex, int) else self.tex_solid(rgb_or_tex)
        return self._c(self.api.mat_diffuse_light(self.h, tex))

    def isotropic(self, rgb_or_tex):
        tex = rgb_or_tex if isinstance(rgb_or_tex, int) else self.tex_solid(rgb_or_tex)
        return self._c(self.api.mat_isotropic(self.h, tex))

    # ---- hittables
    def sphere(self, c, r, mat):
        return self._c(self.api.sphere(self.h, _d3(c), float(r), mat))

    def moving_sphere(self, c0, c1, t0, t1, r, mat):
        return self._c(self.api.moving_sphere(self.h, _d3(c0), _d3(c1), float(t0), float(t1), float(r), mat))

    def gravity_sphere(self, start, t0, r, mat):
        return self._c(self.api.gravity_sphere(self.h, _d3(start), float(t0), float(r), mat))

    def xy_rect(self, x0, x1, y0, y1, k, mat):
        return self._c(self.api.xy_rect(self.h, x0, x1, y0, y1, k, mat))

    def xz_rect(self, x0, x1, z0, z1, k, mat):
        return self._c(self.api.xz_rect(self.h, x0, x1, z0, z1, k, mat))

    def yz_rect(self, y0, y1, z0, z1, k, mat):
        return self._c(self.api.yz_rect(self.h, y0, y1, z0, z1, k, mat))

    def box(self, p0, p1, mat):
        return self._c(self.api.box(self.h, _d3(p0), _d3(p1), mat))

    def triangle(self, v0, v1, v2, mat):
        return self._c(self.api.triangle(self.h, _d3(v0), _d3(v1), _d3(v2), mat))

    def triangle_mesh(self, verts, idx, mat):
        v = np.ascontiguousarray(verts, dtype=np.float64).reshape(-1, 3)
        i = np.ascontiguousarray(idx, dtype=np.uint32).reshape(-1, 3)
        return self._c(self.api.triangle_mesh(self.h, v.ctypes.data_as(c_d3), v.shape[0],
                                              i.ctypes.data_as(C.POINTER(C.c_uint32)), i.shape[0], mat))

    def ply_load(self, path, scale, mat):
        return self._c(self.api.ply_load(self.h, str(path).encode(), float(scale), mat))

    def list(self, ids):
        a = (C.c_int32 * len(ids))(*ids)
        return self._c(self.api.list(self.h, a, len(ids)))

    def bvh(self, ids, t0, t1):
        a = (C.c_int32 * len(ids))(*ids)
        return self._c(self.api.bvh(self.h, a, len(ids), float(t0), float(t1)))

    def translate(self, off, child):
        return self._c(self.api.translate(self.h, _d3(off), child))

    def rotate_y(self, angle_deg, child):
        return self._c(self.api.rotate_y(self.h, float(angle_deg), child))

    def constant_medium(self, rgb, density, boundary):
        return self._c(self.api.constant_medium(self.h, _d3(rgb), float(density), boundary))

    # ---- scene
    def set_root(self, hid):
        return self._c(self.api.scene_set_root(self.h, hid))

    def set_camera(self, lookfrom, lookat, vup, vfov, aspect, aperture, focus, t1, t2):
        return self._c(self.api.scene_set_camera(self.h, _d3(lookfrom), _d3(lookat), _d3(vup), float(vfov),
                                                 float(aspect), float(aperture), float(focus), float(t1), float(t2)))

    def set_camera_fields(self, fields):
        """The 24 f64 fields of the reference's Camera struct (camera.rs:6-17), as its flatten() would pass them."""
        a = (C.c_double * 24)(*[float(x) for x in fields])
        return self._c(self.api.scene_set_camera_fields(self.h, a))

    def set_background(self, rgb):
        return self._c(self.api.scene_set_background(self.h, _d3(rgb)))

    def set_background_gradient(self, horizon_rgb=(1.0, 1.0, 1.0), zenith_rgb=(0.5, 0.7, 1.0)):
        """book-1 sky (the revision of the reference that rendered images/book1.png)"""
        return self._c(self.api.scene_set_background_gradient(self.h, _d3(horizon_rgb), _d3(zenith_rgb)))

    def commit(self):
        return self._c(self.api.scene_commit(self.h))

    def world_build(self, scene_id, seed=0, param=0):
        return self._c(self.api.world_build(self.h, int(scene_id), int(seed), int(param)))

    def num_prims(self):
        return self._c(self.api.scene_num_prims(self.h))

    # ---- product-only controls / diagnostics (librtb200.so; the oracle has neither)
    def set_bvh_builder(self, builder: int):
        """RT_BVH_HOST_SAH = 0 (default) | RT_BVH_DEVICE_LBVH = 1: who builds the BVH at commit (SURVEY.md 8(f) n1)."""
        fn = self.api.lib.rt_scene_set_bvh_builder
        fn.restype, fn.argtypes = C.c_int32, [C.c_void_p, C.c_int32]
        return self._c(fn(self.h, int(builder)))

    def set_bvh_width(self, width: int):
        """0 (auto, default) | 2 | 4: whether rt_scene_commit also builds the 4-wide collapse the fused kernels walk (include/rtb200.h)."""
        fn = self.api.lib.rt_scene_set_bvh_width
        fn.restype, fn.argtypes = C.c_int32, [C.c_void_p, C.c_int32]
        return self._c(fn(self.h, int(width)))

    def bvh_width(self) -> int:
        """rt_scene_bvh_width: 4 if the committed scene carries the 4-wide collapse, else 2."""
        fn = self.api.lib.rt_scene_bvh_width
        fn.restype, fn.argtypes = C.c_int32, [C.c_void_p]
        return self._c(fn(self.h))

    def debug_host_scene(self, nbytes: int):
        """rt_debug_host_scene: the host-flattened DeviceScene as raw bytes (pointers address host arrays owned by the scene).
        Test hook for tests/host_emul; `nbytes` must equal sizeof(DeviceScene)."""
        fn = self.api.lib.rt_debug_host_scene
        fn.restype, fn.argtypes = C.c_int32, [C.c_void_p, C.c_void_p, C.c_uint64]
        buf = C.create_string_buffer(int(nbytes))
        self._c(fn(self.h, buf, int(nbytes)))
        return buf

    def host_check(self):
        """rt_scene_host_check: flattener / BVH invariants + counters of the last commit (include/rtb200.h)."""
        fn = self.api.lib.rt_scene_host_check
        fn.restype, fn.argtypes = C.c_int32, [C.c_void_p, C.POINTER(C.c_int64)]
        out = (C.c_int64 * 16)()
        self._c(fn(self.h, out))
        keys = ("nodes", "max_depth", "main_instances", "instances", "media", "spheres", "movings", "gravities", "rects", "boxes", "tris", "leaves",
                "violations", "prims", "bytes_uploaded", "device_built_prims")
        return dict(zip(keys, [int(x) for x in out]))

    # ---- render / trace
    def image_height(self, cfg: RenderConfig) -> int:
        return self._c(self.api.image_height(C.byref(cfg)))

    def render(self, cfg: RenderConfig, want_accum=False):
        """-> (screen[H,W,3] float64 in Screen layout (row 0 = bottom), accum[H,W,3] int64 | None, stats dict)"""
        H = self.image_height(cfg)
        W = cfg.image_width
        screen = np.zeros((H, W, 3), dtype=np.float64)
        accum = np.zeros((H, W, 3), dtype=np.int64) if want_accum else None
        st = Stats()
        self._c(self.api.render(self.h, C.byref(cfg), screen.ctypes.data_as(c_d3),
                                accum.ctypes.data_as(C.POINTER(C.c_int64)) if want_accum else None, C.byref(st)))
        return screen, accum, st.as_dict()

    def render_multi(self, cfg: RenderConfig, n_gpus: int, shard_mode: int = RT_SHARD_SAMPLES, want_accum=False):
        """rt_render_multi: the same render sharded over n_gpus GPUs by this one process; same return as render()"""
        H = self.image_height(cfg)
        W = cfg.image_width
        screen = np.zeros((H, W, 3), dtype=np.float64)
        accum = np.zeros((H, W, 3), dtype=np.int64) if want_accum else None
        st = Stats()
        self._c(self.api.render_multi(self.h, C.byref(cfg), int(n_gpus), int(shard_mode), screen.ctypes.data_as(c_d3),
                                      accum.ctypes.data_as(C.POINTER(C.c_int64)) if want_accum else None, C.byref(st)))
        return screen, accum, st.as_dict()

    def render_adaptive(self, cfg: RenderConfig, threshold: float, min_samples: int = 64, step: int = 16, radius: int = 1, n_gpus: int = 1):
        """rt_render_adaptive: each pixel rendered until its noise estimate drops below `threshold`, at most cfg.samples_per_pixel
        samples (include/rtb200.h); n_gpus > 1: rt_render_adaptive_multi, the rounds spread over that many GPUs of this box with the
        same results.  -> (screen[H,W,3] float64, accum[H,W,3] int64, samples[H,W] int32, stats dict)"""
        H = self.image_height(cfg)
        W = cfg.image_width
        screen = np.zeros((H, W, 3), dtype=np.float64)
        accum = np.zeros((H, W, 3), dtype=np.int64)
        samples = np.zeros((H, W), dtype=np.int32)
        ac = AdaptiveConfig(int(min_samples), int(step), float(threshold), int(radius))
        st = Stats()
        outs = (screen.ctypes.data_as(c_d3), accum.ctypes.data_as(C.POINTER(C.c_int64)), samples.ctypes.data_as(c_i32p), C.byref(st))
        if n_gpus == 1:
            fn = self.api.lib.rt_render_adaptive
            fn.restype, fn.argtypes = RENDER_ADAPTIVE_SIGNATURE
            self._c(fn(self.h, C.byref(cfg), C.byref(ac), *outs))
        else:
            fn = self.api.lib.rt_render_adaptive_multi
            fn.restype, fn.argtypes = RENDER_ADAPTIVE_MULTI_SIGNATURE
            self._c(fn(self.h, C.byref(cfg), C.byref(ac), int(n_gpus), *outs))
        return screen, accum, samples, st.as_dict()

    def commit_multi(self, n_gpus: int):
        return self._c(self.api.scene_commit_multi(self.h, int(n_gpus)))

    def render_scene_with_time(self, t0, t1, path=None, cfg: RenderConfig = None):
        """render_scene_with_time(t0, t1, path, world)  [ref: world.rs:1249]; cfg None = the reference's 500x500x500spp frame"""
        probe = cfg if cfg is not None else make_config(500, 1.0, 500, 50)
        H, W = self.image_height(probe), probe.image_width
        screen = np.zeros((H, W, 3), dtype=np.float64)
        st = Stats()
        self._c(self.api.render_scene_with_time(self.h, float(t0), float(t1), str(path).encode() if path is not None else None,
                                                C.byref(cfg) if cfg is not None else None, screen.ctypes.data_as(c_d3), C.byref(st)))
        return screen, st.as_dict()

    def trace_batch(self, rays: np.ndarray, t_min=0.001, t_max=float("inf"), flags=RT_TRACE_SKIP_MEDIA, seed=0):
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        out = np.zeros(rays.shape[0], dtype=HIT_DTYPE)
        self._c(self.api.trace_batch(self.h, rays.ctypes.data, rays.shape[0], float(t_min), float(t_max),
                                     int(flags), int(seed), out.ctypes.data))
        return out


def make_rays(o, d, time=0.0) -> np.ndarray:
    o = np.asarray(o, dtype=np.float64).reshape(-1, 3)
    d = np.asarray(d, dtype=np.float64).reshape(-1, 3)
    r = np.zeros(o.shape[0], dtype=RAY_DTYPE)
    r["o"] = o
    r["d"] = d
    r["time"] = time
    return r


def write_ppm_binary(api: Api, path, screen: np.ndarray):
    """P6 fast path of Screen::write_to_ppm_file (product only, SURVEY.md 8(f) n2)."""
    s = np.ascontiguousarray(screen, dtype=np.float64)
    fn = api.lib.rt_write_ppm_binary
    fn.restype, fn.argtypes = C.c_int32, [C.c_char_p, C.c_void_p, C.c_int32, C.c_int32]
    api.check(fn(str(path).encode() if path is not None else None, s.ctypes.data, s.shape[1], s.shape[0]))


def write_ply_binary(api: Api, path, verts: np.ndarray, faces: np.ndarray):
    v = np.ascontiguousarray(verts, dtype=np.float64).reshape(-1, 3)
    f = np.ascontiguousarray(faces, dtype=np.uint32).reshape(-1, 3)
    fn = api.lib.rt_write_ply_binary
    fn.restype, fn.argtypes = C.c_int32, [C.c_char_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]
    api.check(fn(str(path).encode(), v.ctypes.data, v.shape[0], f.ctypes.data, f.shape[0]))


def ply_convert_binary(api: Api, ascii_path, binary_path):
    fn = api.lib.rt_ply_convert_binary
    fn.restype, fn.argtypes = C.c_int32, [C.c_char_p, C.c_char_p]
    api.check(fn(str(ascii_path).encode(), str(binary_path).encode()))


def write_ppm(api: Api, path, screen: np.ndarray):
    s = np.ascontiguousarray(screen, dtype=np.float64)
    H, W = s.shape[0], s.shape[1]
    api.check(api.write_ppm(str(path).encode() if path is not None else None, s.ctypes.data_as(c_d3), W, H))
