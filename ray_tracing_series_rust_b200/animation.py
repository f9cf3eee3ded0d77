"""Animation driver and progressive / checkpointed accumulation (SURVEY.md 8(f) n4).

The reference has the per-frame entry `render_scene_with_time(t0, t1, path, world)` (src/world.rs:1249-1330) but
not the loop around it (its `/video_testing/` driver is absent from the repo), and a 10 000-spp still
(`README.md`: 12 453 s) is one uninterruptible call.  This module supplies both on top of the C-ABI:

* `AnimationDriver`   frame f -> rank f mod world (`sharding.frames_for_rank`), per frame: shutter window ->
                      `rt_scene_set_camera` + `rt_scene_commit` (GravitySphere windows, BVH) -> render -> PPM
                      (P3 as the reference, or P6).  Finished frames are skipped on restart.
* `ProgressiveRender` one still rendered as sample ranges `[s0, s1)` (rt_render_config.sample_begin / sample_end)
                      summed into the int64 accumulator, with an atomic single-file checkpoint every few chunks.  Philox
                      streams are keyed by the global sample index and the sum is integer, so a render that
                      was interrupted and resumed is bit-identical to the one-shot render.
* `resolve_accumulator`  host mirror of `k_resolve` (Vec3::get_normalized_color, src/vec3.rs:89-107), also with per-pixel
                         sample counts (`k_resolve_adaptive`).
"""
from __future__ import annotations

import json
import os
from typing import Callable, Iterable, Optional, Sequence

import numpy as np

from . import capi, sharding


def resolve_accumulator(accum: np.ndarray, spp, rendered_rows: Optional[int] = None) -> np.ndarray:
    """int64 fixed-point (2^32) radiance sums [H, W, 3] -> the reference's Screen (integer-valued f64, row 0 = bottom).

    `spp` is one sample count for every pixel, or per-pixel counts [H, W] (rt_render_adaptive's samples; a pixel with 0 samples
    resolves to black)."""
    s = accum.astype(np.float64) * (1.0 / 4294967296.0)
    if np.ndim(spp) == 0:
        scale = 1.0 / float(spp)
    else:
        with np.errstate(divide="ignore"):
            scale = (1.0 / np.asarray(spp, dtype=np.float64))[..., None]
    with np.errstate(invalid="ignore"):
        c = np.sqrt(s * scale)
    c = np.where(c < 0.0, 0.0, np.where(c > 1.0, 1.0, c))  # mutil.rs:1-9
    q = 255.9 * c
    out = np.where(np.isnan(q), 0.0, np.trunc(q))          # `as i32`
    if rendered_rows is not None:
        out[rendered_rows:] = 0.0                          # compat_threads remainder rows (world.rs:1198-1202)
    return out


class ProgressiveRender:
    """Accumulate `spp_total` samples in chunks with resumable checkpoints.

    `render_chunk(s0, s1) -> int64 array [H, W, 3]` renders samples [s0, s1) of every pixel (for a scene:
    `lambda a, b: scene.render(make_config(..., spp_total, ..., sample_begin=a, sample_end=b), want_accum=True)[1]`).
    """

    def __init__(self, render_chunk: Callable[[int, int], np.ndarray], shape: Sequence[int], spp_total: int, chunk: int,
                 checkpoint: Optional[str] = None, every: int = 1, meta: Optional[dict] = None):
        if spp_total < 1 or chunk < 1 or every < 1:
            raise ValueError("bad progressive request")
        self.render_chunk, self.shape, self.spp_total, self.chunk = render_chunk, tuple(shape), int(spp_total), int(chunk)
        self.checkpoint, self.every = checkpoint, int(every)
        self.meta = dict(meta or {})
        self.accum = np.zeros(self.shape, dtype=np.int64)
        self.done = 0
        if checkpoint and os.path.exists(self._file()):
            self._load()

    # ---- checkpoint = ONE file <path>.npz holding the accumulator, the number of samples it contains and the identity of the
    # render; written to a temporary and renamed, so a crash at any point leaves either the old or the new checkpoint, never an
    # accumulator paired with another checkpoint's sample count (which would add a sample range twice on resume)
    def _file(self):
        return self.checkpoint + ".npz"

    def _identity(self):
        return {"shape": list(self.shape), "spp_total": self.spp_total, "meta": self.meta}

    def _load(self):
        with np.load(self._file(), allow_pickle=False) as z:
            ident = json.loads(str(z["identity"]))
            a, done = z["accum"], int(z["samples_done"])
        if ident != self._identity():
            raise ValueError("checkpoint belongs to a different render: %r" % (ident,))
        if a.shape != self.shape or a.dtype != np.int64 or not (0 <= done <= self.spp_total):
            raise ValueError("corrupt checkpoint")
        self.accum, self.done = a, done

    def save(self):
        if not self.checkpoint:
            return
        tmp = self.checkpoint + ".tmp.npz"
        with open(tmp, "wb") as f:
            np.savez(f, accum=self.accum, samples_done=np.int64(self.done), identity=np.array(json.dumps(self._identity(), sort_keys=True)))
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, self._file())

    def run(self, max_chunks: Optional[int] = None) -> np.ndarray:
        """Renders until spp_total (or for `max_chunks` chunks); returns the accumulator so far."""
        n = 0
        while self.done < self.spp_total and (max_chunks is None or n < max_chunks):
            s1 = min(self.spp_total, self.done + self.chunk)
            part = self.render_chunk(self.done, s1)
            if part.shape != self.shape or part.dtype != np.int64:
                raise ValueError("render_chunk must return the int64 accumulator of the chunk")
            self.accum += part
            self.done = s1
            n += 1
            if n % self.every == 0 or self.done == self.spp_total:
                self.save()
        return self.accum

    @property
    def finished(self) -> bool:
        return self.done >= self.spp_total

    def screen(self) -> np.ndarray:
        """The image of the samples accumulated so far (a preview until `finished`)."""
        return resolve_accumulator(self.accum, max(self.done, 1))


def progressive_scene_render(scene: "capi.Scene", width: int, aspect: float, spp_total: int, max_depth: int, seed: int = 1, chunk: int = 100,
                             checkpoint: Optional[str] = None, every: int = 1, flags: int = 0) -> ProgressiveRender:
    """ProgressiveRender over one committed scene (single GPU; for several, give each rank its `sharding.sample_range`)."""
    cfg0 = capi.make_config(width, aspect, spp_total, max_depth, seed=seed)
    H = scene.image_height(cfg0)

    def chunk_fn(s0, s1):
        cfg = capi.make_config(width, aspect, spp_total, max_depth, seed=seed, sample_begin=s0, sample_end=s1, flags=flags)
        return scene.render(cfg, want_accum=True)[1]

    return ProgressiveRender(chunk_fn, (H, width, 3), spp_total, chunk, checkpoint, every,
                             meta={"width": width, "aspect": aspect, "max_depth": max_depth, "seed": seed})


class AnimationDriver:
    """The loop around render_scene_with_time: one PPM per frame, frames dealt round-robin to ranks.

    `shutter(f) -> (t0, t1)`; `camera` = the nine Camera::new arguments without the two times (the reference's
    frame camera is lookfrom (13,2,3), lookat 0, vup y, vfov 20, aspect, aperture 0.1, focus 10: world.rs:1259-1274).
    Re-running skips frames whose file already exists (frame-granular checkpoint)."""

    def __init__(self, scene: "capi.Scene", width: int, aspect: float, spp: int, max_depth: int, out_pattern: str,
                 shutter: Callable[[int], Sequence[float]] = lambda f: (0.4 * f, 0.4 * f + 0.4),
                 camera=((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, None, 0.1, 10.0), seed: int = 5, binary: bool = False,
                 rank: int = 0, world: int = 1, resume: bool = True):
        self.scene, self.width, self.aspect, self.spp, self.max_depth = scene, int(width), float(aspect), int(spp), int(max_depth)
        self.out_pattern, self.shutter, self.seed, self.binary = out_pattern, shutter, int(seed), bool(binary)
        cam = list(camera)
        if cam[4] is None:
            cam[4] = self.aspect
        self.camera = cam
        self.rank, self.world, self.resume = int(rank), int(world), bool(resume)

    def frame_path(self, f: int) -> str:
        return self.out_pattern % f

    def frames(self, n_frames: int):
        return sharding.frames_for_rank(n_frames, self.rank, self.world)

    def render_frame(self, f: int):
        t0, t1 = self.shutter(f)
        lookfrom, lookat, vup, vfov, aspect, aperture, focus = self.camera
        self.scene.set_camera(lookfrom, lookat, vup, vfov, aspect, aperture, focus, float(t0), float(t1))
        self.scene.commit()  # re-derives GravitySphere windows and bounds for this shutter
        cfg = capi.make_config(self.width, self.aspect, self.spp, self.max_depth, seed=self.seed + f)
        screen, _, st = self.scene.render(cfg)
        path = self.frame_path(f)
        tmp = path + ".part"
        (capi.write_ppm_binary if self.binary else capi.write_ppm)(self.scene.api, tmp, screen)
        os.replace(tmp, path)
        return screen, st

    def run(self, n_frames: int, frames: Optional[Iterable[int]] = None):
        """-> list of (frame, path, stats | None); stats None = skipped because the file was already there."""
        out = []
        for f in (self.frames(n_frames) if frames is None else frames):
            path = self.frame_path(f)
            if self.resume and os.path.exists(path):
                out.append((f, path, None))
                continue
            _, st = self.render_frame(f)
            out.append((f, path, st))
        return out
