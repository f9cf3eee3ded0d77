"""The 4-wide sphere kernels of the fused mode (k_mega, WIDE): one build for scenes without Noise / Image textures, compiled for
RT_MEGA_OCC_SPH CTAs per SM, and one with the full texture code for the others.

On the CPU: the shipped instantiations fit their register budget without spilling (the ptxas -v log csrc/Makefile writes next to the
object).  On the GPU: each build renders, bit for bit, what the wavefront renders for the same scene.
"""
import os
import re

import numpy as np
import pytest

import ray_tracing_series_rust_b200 as rtb
from ray_tracing_series_rust_b200 import capi

LOG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ray_tracing_series_rust_b200", "csrc", "build",
                   "kernels.ptxas.log")


def _wide_sphere_kernels():
    """{(primitive mask, full textures): (CTAs per SM, registers, spill store bytes, spill load bytes)} from the ptxas log."""
    text = open(LOG).read()
    out = {}
    # k_mega<MEDIA = false, OCC, GENERAL_MEDIA = false, PM, XF = false, WIDE = true, FULLTEX>
    for m in re.finditer(r"Function properties for _ZN3rtb6k_megaILb0ELi(\d+)ELb0ELj(\d+)ELb0ELb1ELb([01])E\S*\n"
                         r"\s*(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\n"
                         r"ptxas info\s*: Used (\d+) registers", text):
        occ, pm, full, _, st, ld, regs = (int(x) for x in m.groups())
        out[(pm, bool(full))] = (occ, regs, st, ld)
    return out


@pytest.mark.skipif(not os.path.exists(LOG), reason="needs the library built by csrc/Makefile (build/kernels.ptxas.log)")
def test_wide_sphere_kernels_fit_their_occupancy_without_spills():
    k = _wide_sphere_kernels()
    for pm in (0x1, 0x3, 0x5):
        assert (pm, False) in k and (pm, True) in k, sorted(k)
    for pm in (0x1, 0x5):  # book-1 final, the bouncing-spheres animation
        occ, regs, st, ld = k[(pm, False)]
        assert occ >= 6, (pm, occ)
        assert regs * 128 * occ <= 65536, (pm, regs, occ)
        assert st == 0 and ld == 0, (pm, st, ld)


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id", [0, 1, 2, 13, 8, 99])
def test_wide_sphere_kernels_match_the_wavefront(scene_id):
    # 0 checker texture, 13 book-1 final (solid colours): the slim build; 1 Perlin spheres, 2 image texture: the full-texture build;
    # 8 gravity spheres, 99 moving spheres (book-1 as shipped): the other two primitive masks.  Forced fused mode on the 4-wide tree
    # against forced wavefront mode on the sibling pairs: same accumulator, same segment count
    aspect = 16 / 9 if scene_id == 99 else 1.5
    acc, segs = {}, {}
    for width, flags in ((4, 8), (2, 4)):  # RT_RENDER_FORCE_FUSED, RT_RENDER_FORCE_WAVEFRONT
        g = rtb.new_scene()
        g.world_build(scene_id, 0xB001, 0)
        g.set_bvh_width(width)
        g.commit()
        _, acc[width], st = g.render(capi.make_config(80, aspect, 6, 50, seed=11, flags=flags), want_accum=True)
        segs[width] = st["segments"]
        g.close()
    assert np.array_equal(acc[4], acc[2]) and segs[4] == segs[2]
    assert acc[4].any()
