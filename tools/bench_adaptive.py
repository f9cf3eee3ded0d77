"""Adaptive sampling against fixed sample counts on one GPU or several (not part of the product; bench.py is the headline benchmark).

    python tools/bench_adaptive.py [--out FILE] [--reps 3] [--thresholds 0.02,0.05,0.1,0.2,0.5] [--step 16] [--gpus 1] [--profile-checks]

For book-2 final (scene 6, 1000x1000, max 2000 spp) and book-1 final (scene 13, 800x533, max 500 spp): rt_render at max, then
rt_render_adaptive (min_samples 64, step 16 or --step, radius 1) at each threshold.  Per run: min / median / max wall ms of `reps` calls (host clock around
the call, which ends in a stream synchronise; the fixed render and the thresholds alternate within each repetition), mean samples per pixel, rounds, paths/s, and the RMSE of the image against an
independent-seed rt_render at max: on the Screen (0..255) and on the linear radiance (sum / samples).  The reference has noise of its
own, so a fixed render at max is the floor the adaptive rows compare with.  frac_stopped_zero / sq_err_share_stopped_zero: the
pixels that stopped before max with all-zero sums, and their share of the Screen's squared error.  The card's name and power limit come from the same run.
--gpus N > 1: the fixed render is rt_render_multi and the adaptive rows rt_render_adaptive_multi over N GPUs.  accum_sha / samples_sha:
hashes of the accumulator and the sample counts, to compare builds and GPU counts (they must not change).  --profile-checks: one more
call per threshold under torch.profiler; ms_checks_device = the device time of the check points (error, dilation, compaction, list
copies; staged peer copies included), which the timed calls do not see.
One JSON line per row, also written to --out.
"""
import hashlib
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


def device_count():
    import torch
    return torch.cuda.device_count()


def sha(x):
    return hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()[:16]


def checks_device_ms(call):
    """Device time of everything a call runs besides its render rounds and its resolve: the check kernels (k_adaptive_*), CUB's
    compaction and the device-to-device copies (pixel lists, staged peer accumulators)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
    total = 0.0
    for ev in prof.events():
        name = ev.name
        if ev.device_type.name != "CUDA":
            continue
        check = ("k_adaptive_error" in name or "k_adaptive_keep" in name or "DeviceSelect" in name or "DeviceCompact" in name
                 or ("Memcpy" in name and ("PtoP" in name or "DtoD" in name)))
        if check:
            total += ev.device_time
    return round(total / 1e3, 2)


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
    ap.add_argument("--gpus", type=int, default=1, help="GPUs of this box to spread every render over")
    ap.add_argument("--profile-checks", action="store_true", help="device time of the check points, from one profiled call per threshold")
    a = ap.parse_args()
    STEP = a.step
    taus = [float(x) for x in a.thresholds.split(",")]
    rows = []

    def emit(d):
        rows.append(d)
        print(json.dumps(d), flush=True)

    emit({"card": card(), "device_count": device_count(), "gpus": a.gpus, "lib": os.path.basename(rtb.LIB_PATH), "min_samples": MIN_SAMPLES,
          "step": STEP, "radius": RADIUS})

    def fixed(cfg, want_accum=False):
        return g.render(cfg, want_accum=want_accum) if a.gpus == 1 else g.render_multi(cfg, a.gpus, want_accum=want_accum)

    def adaptive_run(cfg, tau, min_samples=MIN_SAMPLES):
        return g.render_adaptive(cfg, tau, min_samples=min_samples, step=STEP, radius=RADIUS, n_gpus=a.gpus)

    for name in a.scenes.split(","):
        sid, seed, W, aspect, spp = SCENES[name]
        g = rtb.new_scene()
        g.world_build(sid, seed, 0)
        g.commit()
        cfg = capi.make_config(W, aspect, spp, 50, seed=1)
        H = g.image_height(cfg)
        fixed(capi.make_config(W, aspect, 8, 50, seed=1))  # warm-up: modules, workspace, output buffers, replicas
        adaptive_run(capi.make_config(W, aspect, 64, 50, seed=1), 0.05, min_samples=0)
        ref_screen, ref_acc, _ = g.render(capi.make_config(W, aspect, spp, 50, seed=1001), want_accum=True)  # independent seed
        ref_lin = linear(ref_acc, spp)

        # the fixed render and every threshold alternate within each repetition, so drift of the shared machine hits all of them alike
        runs = [None] + taus
        times = {t: [] for t in runs}
        res = {}
        for _ in range(a.reps):
            for tau in runs:
                t0 = time.perf_counter()
                res[tau] = fixed(cfg, want_accum=True) if tau is None else adaptive_run(cfg, tau)
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
                        "speedup_median": round(fixed_med / float(np.median(ms)), 3), "accum_sha": sha(acc), "samples_sha": sha(smp)})
            if a.profile_checks and tau is not None:
                row["ms_checks_device"] = checks_device_ms(lambda: adaptive_run(cfg, tau))
            emit(row)
        g.close()
    if a.out:
        with open(a.out, "w") as f:
            for d in rows:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
