"""The quality cases of tests/test_denoise.py (and book-1 final 800x533 at 500 spp) over a grid of filter settings (not part of the product).

    python tools/sweep_denoise.py > profiles/denoise_sweep_b200.jsonl

Per case: an independent-seed rt_render reference, the raw render, then rt_render_denoised at every sigma_color, iterations,
sigma_normal (sigma_albedo 0.1) and aov_samples of the grid; one JSON line per setting with the linear RMSE ratio denoised / raw.
"""
import json, sys, os, itertools
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import ray_tracing_series_rust_b200 as rtb
from ray_tracing_series_rust_b200 import capi
S = 4294967296.0
CASES = [(13, 0, 1.5, 400, 16, 1024), (4, 0, 1.0, 300, 16, 1024), (14, 48, 1.0, 256, 16, 1024), (5, 0, 1.0, 200, 16, 1024),
         (6, 0, 1.0, 200, 16, 1024), (13, 0, 1.5, 200, 1024, 8192), (13, 0, 1.5, 800, 500, 8192)]
for sid, param, aspect, W, spp, rspp in CASES:
    g = rtb.new_scene(); g.world_build(sid, 3 if W != 800 else 0xB001, param); g.commit()
    ref = g.render(capi.make_config(W, aspect, rspp, 50, seed=1000 + sid), want_accum=True)[1] / S / rspp
    acc = g.render(capi.make_config(W, aspect, spp, 50, seed=7), want_accum=True)[1]
    raw = float(np.sqrt(np.mean((acc / S / spp - ref) ** 2)))
    for sc, its, sn, m in itertools.product((0.5, 1.0, 1.5, 2.0, 3.0, 4.0), (2, 3, 4, 5), (0.125, 0.25), (8, 16)):
        if m > spp: continue
        lin = g.render_denoised(capi.make_config(W, aspect, spp, 50, seed=7), aov_samples=m, iterations=its, sigma_color=sc, sigma_albedo=0.1, sigma_normal=sn)[1]
        r = float(np.sqrt(np.mean((lin - ref) ** 2))) / raw
        print(json.dumps({"scene": sid, "W": W, "spp": spp, "sc": sc, "its": its, "sn": sn, "m": m, "ratio": round(r, 4)}), flush=True)
    g.close()
