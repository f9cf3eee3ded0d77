"""Denoised renders against raw renders on one GPU (not part of the product; bench.py is the headline benchmark).

    python tools/bench_denoise.py [--out FILE] [--reps 3] [--sweep]

For book-1 final (scene 13, 800x533) at 16, 64 and 500 spp and book-2 final (scene 6, 1000x1000) at 64 spp: rt_render against
rt_render_denoised with the default settings (aov_samples min(8, spp), 5 iterations, sigma_color 4, sigma_albedo 0.1, sigma_normal
0.125).  Per row: min / median wall ms of `reps` calls of each (host clock around the call, which ends in a stream synchronise; the two
alternate), the device time of the feature pass (k_aov) and of the filter kernels (k_dn_*) from one more call under torch.profiler, and
the linear RMSE (sum / samples) of the raw and the denoised image against an independent-seed rt_render at `ref_spp`.  For the 16-spp
rows, raw_spp_matching = the raw sample count whose RMSE equals the denoised one (log-log interpolation between raw renders at 16 .. 1024
spp).  --sweep: the denoised RMSE of book-1 final at 16 spp over a small grid of sigmas and iteration counts.  The card's name and power
limit come from the same run.  One JSON line per row, also written to --out.
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

SCENES = {  # name: (scene id, scene seed, width, aspect, spp list, reference spp)
    "book1_final": (13, 0xB001, 800, 1.5, (16, 64, 500), 8192),
    "book2_final": (6, 0xB002, 1000, 1.0, (64,), 4096),
}
MATCH_SPP = (16, 32, 64, 128, 256, 512, 1024)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def rmse(a, b):
    return float(np.sqrt(np.mean((np.asarray(a, np.float64) - np.asarray(b, np.float64)) ** 2)))


def kernel_ms(call):
    """device ms of the feature pass and of the filter kernels in one call, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
    aov = filt = 0.0
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        if "k_aov" in ev.name:
            aov += ev.device_time
        elif "k_dn_" in ev.name:
            filt += ev.device_time
    return round(aov / 1e3, 3), round(filt / 1e3, 3)


def matching_spp(curve, target):
    """raw spp whose RMSE equals `target`, log-log interpolation over (spp, rmse) pairs; None if outside"""
    for (s0, r0), (s1, r1) in zip(curve, curve[1:]):
        if r0 >= target >= r1:
            t = (np.log(r0) - np.log(target)) / (np.log(r0) - np.log(r1))
            return round(float(np.exp(np.log(s0) + t * (np.log(s1) - np.log(s0)))), 1)
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scenes", default="book1_final,book2_final")
    ap.add_argument("--sweep", action="store_true")
    a = ap.parse_args()
    rows = []

    def emit(d):
        rows.append(d)
        print(json.dumps(d), flush=True)

    emit({"card": card(), "lib": os.path.basename(rtb.LIB_PATH)})
    for name in a.scenes.split(","):
        sid, seed, W, aspect, spps, ref_spp = SCENES[name]
        g = rtb.new_scene()
        g.world_build(sid, seed, 0)
        g.commit()
        g.render(capi.make_config(W, aspect, 8, 50, seed=1))  # warm-up: modules, workspace, buffers
        g.render_denoised(capi.make_config(W, aspect, 8, 50, seed=1))
        t0 = time.perf_counter()
        ref = g.render(capi.make_config(W, aspect, ref_spp, 50, seed=1001), want_accum=True)[1] / 4294967296.0 / ref_spp  # independent seed
        emit({"scene": name, "ref_spp": ref_spp, "ref_ms": round((time.perf_counter() - t0) * 1e3, 1)})
        curve = None
        for spp in spps:
            cfg = capi.make_config(W, aspect, spp, 50, seed=1)
            t_raw, t_den = [], []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                _, acc, _ = g.render(cfg, want_accum=True)
                t_raw.append((time.perf_counter() - t0) * 1e3)
                t0 = time.perf_counter()
                _, lin, acc_d, st = g.render_denoised(cfg)
                t_den.append((time.perf_counter() - t0) * 1e3)
            assert np.array_equal(acc, acc_d), "rt_render_denoised's accumulator must be rt_render's"
            aov_ms, filt_ms = kernel_ms(lambda: g.render_denoised(cfg))
            raw_e, den_e = rmse(acc / 4294967296.0 / spp, ref), rmse(lin, ref)
            row = {"scene": name, "W": W, "H": acc.shape[0], "spp": spp, "aov_samples": min(8, spp),
                   "render_ms_min": round(min(t_raw), 2), "render_ms_median": round(float(np.median(t_raw)), 2),
                   "denoised_ms_min": round(min(t_den), 2), "denoised_ms_median": round(float(np.median(t_den)), 2),
                   "aov_device_ms": aov_ms, "filter_device_ms": filt_ms,
                   "rmse_raw": round(raw_e, 6), "rmse_denoised": round(den_e, 6), "ratio": round(den_e / raw_e, 4)}
            if spp == 16:
                if curve is None:
                    curve = [(s, rmse(g.render(capi.make_config(W, aspect, s, 50, seed=1), want_accum=True)[1] / 4294967296.0 / s, ref)) for s in MATCH_SPP]
                    emit({"scene": name, "raw_rmse_curve": [[s, round(e, 6)] for s, e in curve]})
                row["raw_spp_matching"] = matching_spp(curve, den_e)
            emit(row)
        if a.sweep and name == "book1_final":
            cfg = capi.make_config(W, aspect, 16, 50, seed=1)
            raw_e = rmse(g.render(cfg, want_accum=True)[1] / 4294967296.0 / 16, ref)
            for sc in (2.0, 4.0, 8.0):
                for sa in (0.05, 0.1, 0.2):
                    for sn in (0.125, 0.25):
                        for its in (4, 5):
                            lin = g.render_denoised(cfg, iterations=its, sigma_color=sc, sigma_albedo=sa, sigma_normal=sn)[1]
                            emit({"sweep": name, "spp": 16, "iterations": its, "sigma_color": sc, "sigma_albedo": sa, "sigma_normal": sn,
                                  "ratio": round(rmse(lin, ref) / raw_e, 4)})
        g.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
