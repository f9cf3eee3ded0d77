"""Adaptive sampling against fixed sample counts on one GPU (not part of the product; bench.py is the headline benchmark).

    python tools/bench_adaptive.py [--out FILE] [--reps 3] [--thresholds 0.02,0.05,0.1,0.2,0.5] [--step 16]

For book-2 final (scene 6, 1000x1000, max 2000 spp) and book-1 final (scene 13, 800x533, max 500 spp): rt_render at max, then
rt_render_adaptive (min_samples 64, step 16 or --step, radius 1) at each threshold.  Per run: min / median / max wall ms of `reps` calls (host clock around
the call, which ends in a stream synchronise; the fixed render and the thresholds alternate within each repetition), mean samples per pixel, rounds, paths/s, and the RMSE of the image against an
independent-seed rt_render at max: on the Screen (0..255) and on the linear radiance (sum / samples).  The reference has noise of its
own, so a fixed render at max is the floor the adaptive rows compare with.  frac_stopped_zero / sq_err_share_stopped_zero: the
pixels that stopped before max with all-zero sums, and their share of the Screen's squared error.  The card's name and power limit come from the same run.
One JSON line per row, also written to --out.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import ray_tracing_series_rust_b200 as rtb  # noqa: E402
from ray_tracing_series_rust_b200 import capi  # noqa: E402

SCENES = {  # name: (scene id, scene seed, width, aspect, max spp)
    "book2_final": (6, 0xB002, 1000, 1.0, 2000),
    "book1_final": (13, 0xB001, 800, 1.5, 500),
}
MIN_SAMPLES, RADIUS = 64, 1


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def linear(accum, samples):
    n = np.asarray(samples, dtype=np.float64)
    if n.ndim:
        n = n[..., None]
    return accum.astype(np.float64) / 4294967296.0 / np.maximum(n, 1.0)


def rmse(a, b):
    return float(np.sqrt(np.mean((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scenes", default="book2_final,book1_final")
    ap.add_argument("--thresholds", default="0.02,0.05,0.1,0.2,0.5")
    ap.add_argument("--step", type=int, default=16, help="samples per round")
    a = ap.parse_args()
    STEP = a.step
    taus = [float(x) for x in a.thresholds.split(",")]
    rows = []

    def emit(d):
        rows.append(d)
        print(json.dumps(d), flush=True)

    emit({"card": card(), "min_samples": MIN_SAMPLES, "step": STEP, "radius": RADIUS})
    for name in a.scenes.split(","):
        sid, seed, W, aspect, spp = SCENES[name]
        g = rtb.new_scene()
        g.world_build(sid, seed, 0)
        g.commit()
        cfg = capi.make_config(W, aspect, spp, 50, seed=1)
        H = g.image_height(cfg)
        g.render(capi.make_config(W, aspect, 8, 50, seed=1))  # warm-up: modules, workspace, output buffers
        g.render_adaptive(capi.make_config(W, aspect, 64, 50, seed=1), 0.05, min_samples=0, step=STEP, radius=RADIUS)
        ref_screen, ref_acc, _ = g.render(capi.make_config(W, aspect, spp, 50, seed=1001), want_accum=True)  # independent seed
        ref_lin = linear(ref_acc, spp)

        # the fixed render and every threshold alternate within each repetition, so drift of the shared machine hits all of them alike
        runs = [None] + taus
        times = {t: [] for t in runs}
        res = {}
        for _ in range(a.reps):
            for tau in runs:
                t0 = time.perf_counter()
                if tau is None:
                    res[tau] = g.render(cfg, want_accum=True)
                else:
                    res[tau] = g.render_adaptive(cfg, tau, min_samples=MIN_SAMPLES, step=STEP, radius=RADIUS)
                times[tau].append((time.perf_counter() - t0) * 1e3)
        fixed_med = float(np.median(times[None]))
        for tau in runs:
            ms = np.array(times[tau])
            row = {"scene": name, "W": W, "H": H, "max_spp": spp, "threshold": tau, "reps": a.reps, "wall_ms_min": round(float(ms.min()), 1),
                   "wall_ms_median": round(float(np.median(ms)), 1), "wall_ms_max": round(float(ms.max()), 1)}
            if tau is None:
                screen, acc, st = res[tau]
                smp = np.full((H, W), spp, np.int32)
            else:
                screen, acc, smp, st = res[tau]
                assert st["paths"] == int(smp.sum())
            err2 = ((screen - ref_screen) ** 2).sum(axis=2)
            # pixels that stopped early although neither half saw any light (err = 0): their share of the Screen's squared error
            zero = (smp < spp) & ~acc.any(axis=2)
            row.update({"ms_device": round(st["ms_device"], 1), "mean_spp": round(float(smp.mean()), 2), "frac_at_max": round(float((smp == spp).mean()), 4),
                        "rounds": int(-(-int(smp.max()) // STEP)) if tau is not None else 1, "paths": st["paths"],
                        "Gpaths_s": round(st["paths"] / float(np.median(ms)) / 1e6, 3), "rmse_screen": round(rmse(screen, ref_screen), 4),
                        "rmse_linear": round(rmse(linear(acc, smp), ref_lin), 6), "frac_stopped_zero": round(float(zero.mean()), 4),
                        "sq_err_share_stopped_zero": round(float(err2[zero].sum() / max(err2.sum(), 1e-30)), 4),
                        "speedup_median": round(fixed_med / float(np.median(ms)), 3)})
            emit(row)
        g.close()
    if a.out:
        with open(a.out, "w") as f:
            for d in rows:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
