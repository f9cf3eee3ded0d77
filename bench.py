#!/usr/bin/env python
"""bench.py — paths/s of the B200 path-tracing hot path on the reference's headline configs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload book1_final] [--impl reference] [--dump-outputs DIR]

A "step" is one complete render of the workload (every pixel, every sample, depth 50) through
librtb200.so.  `value` = camera paths per second over all ranks with the scene already resident in
HBM; `e2e` = the same through the host-buffer plugin call a Rust host would make - rt_scene_commit
(flatten + BVH build + H2D upload) + rt_render(host Screen buffer) at N = 1, rt_scene_commit_multi +
rt_render_multi (one process driving all N GPUs, peer-memory reduce + resolve) at N > 1 - with every
copy inside the timed region.

Multi-GPU (torchrun, one rank per GPU): STRONG scaling by default - the workload's own spp (500 for
book-1 final) is split into N sample ranges of ONE image (Philox streams are keyed by the global sample
index), the int64 accumulators are summed with one NCCL reduce to rank 0, which resolves the image; the
line also carries `also.book2_final_strong`, the full 10 000-spp book-2 final split the same way.
--scaling weak renders the full spp on every rank (an N x spp image).

--impl reference times the CPU restatement of the reference (oracle/, all host threads) on a bounded
sample of the same workload: the reference itself is Rust and cannot be built in this image.

--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (see dump_outputs).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

# name: (scene id, scene seed, param, width, aspect, spp, depth, camera override | None, description)
WORKLOADS = {
    "book1_final": (13, 0xB001, 0, 800, 1.5, 500, 50, None,
                    "RTIOW book-1 final random spheres 800x533, 500 spp, depth 50 (BASELINE configs[0], README.md:11-23)"),
    "book1_shipped": (99, 0xB001, 0, 800, 1.5, 500, 50, None,
                      "gen_random_scene as shipped (checker ground, moving spheres, 16/9 camera) 800x533, 500 spp"),
    "cornell_smoke": (5, 0xB002, 0, 600, 1.0, 1000, 50, None, "Cornell box with constant-medium smoke boxes 600x600, 1000 spp (BASELINE configs[1])"),
    "book2_final": (6, 0xB002, 0, 1000, 1.0, 10000, 50, None, "Next Week final scene 1000x1000, 10000 spp (BASELINE configs[2])"),
    "mesh_room": (14, 0xB004, 660, 1000, 1.0, 1000, 50, None, "synthetic dragon-scale PLY mesh (871200 tris) room 1000x1000, 1000 spp (BASELINE configs[3])"),
    "bouncing_anim": (8, 0xB005, 240, 800, 1.5, 200, 50, None,
                      "bouncing-spheres motion-blur animation, 240 frames 800x533 @ 200 spp, shutter [0.4f, 0.4f+0.4), frames sharded across GPUs (BASELINE configs[4])"),
}
README_BOOK1_10T_PATHS_PER_S = 800 * 533 * 500 / 146.440  # README.md:23 "Parallel; 10 threads" 146.440 s (unspecified CPU)

# SURVEY.md §8(d) accounting constants (bytes, device f32 layout)
B_NODE, B_STATE = 32, 160
B_PRIM = {0: 16, 1: 32, 2: 20, 3: 24, 4: 24, 5: 48, 6: 8}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_scene(mod, new_scene, wl):
    sid, seed, param, W, aspect, spp, depth, cam, _ = wl
    s = new_scene()
    s.world_build(sid, seed, param)
    if cam:
        s.set_camera(*cam)
    return s


DUMP_BYTES_MAX = 64_000_000


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes every array as out_dir/<name>.npy, so that two builds can be compared output for output (a step's
    seed depends only on its index, so the same arguments render the same paths).  Rendering modes write rank 0's results:
      screen  (H, W, 3) float64  the resolved Screen, row 0 = bottom, every value an integer 0..255
      accum   (H, W, 3) float64  the summed int64 fixed-point accumulator (units of 2^-32), exact below 2^53; not with the peer group
    bouncing_anim writes screen_frameNNN (float32, exact for 0..255) for up to 8 evenly spaced frames of rank 0."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES_MAX:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes, more than {DUMP_BYTES_MAX}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print(f"[bench] wrote {', '.join(sorted(arrays))} ({total / 1e6:.1f} MB) to {out_dir}", file=sys.stderr, flush=True)


def oracle_counts_per_segment(st):
    """algorithmic bytes per segment from the oracle's event counters (SURVEY.md §8d formula)."""
    seg = max(st["segments"], 1)
    v = st["box_tests"] / seg
    prim_bytes = sum(B_PRIM[t] * st["prim_tests"][t] for t in range(7)) / seg
    return {"box_tests_per_segment": v, "prim_tests_per_segment": sum(st["prim_tests"]) / seg, "segments_per_path": st["segments"] / max(st["paths"], 1),
            "bytes_per_segment": B_NODE * v + prim_bytes + B_STATE}


def run_cpu_sample(wl, target_s, threads, seed=1, width=None):
    """Times the oracle (all host threads) on a bounded sample: the full image (or, with `width`, the same view at a lower
    resolution) at a reduced spp."""
    import oracle
    from ray_tracing_series_rust_b200 import capi
    sid, sseed, param, W, aspect, spp, depth, cam, desc = wl
    full_W = W
    W = width or W
    s = build_scene(oracle, oracle.new_scene, wl)
    s.commit()
    # calibrate with 1 spp, then pick the spp that fills ~target_s
    t0 = time.time()
    _, _, st = s.render(capi.make_config(W, aspect, 1, depth, seed=seed, threads=threads))
    rate = st["paths"] / max(time.time() - t0, 1e-6)
    H = s.image_height(capi.make_config(W, aspect, 1, depth))
    use = max(1, min(spp, int(rate * target_s / (W * H))))
    t0 = time.time()
    _, _, st = s.render(capi.make_config(W, aspect, use, depth, seed=seed, threads=threads))
    dt = time.time() - t0
    return {"paths_per_s": st["paths"] / dt, "seconds": dt, "spp": use, "stats": st,
            "sample": f"{'full' if W == full_W else 'same view at'} {W}x{H} image at {use} of {spp} spp, depth {depth} ({st['paths']} paths, {dt:.1f} s)"}


def reference_arm(args, wl, name):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    per_step = max(2.0, min(12.0, 150.0 / max(1, args.steps + args.warmup)))
    vals = []
    last = None
    for i in range(args.warmup + args.steps):
        last = run_cpu_sample(wl, per_step, threads, seed=1 + i)
        if i >= args.warmup:
            vals.append(last)
    tot_paths = sum(v["stats"]["paths"] for v in vals)
    tot_s = sum(v["seconds"] for v in vals)
    value = tot_paths / tot_s
    out = {
        "impl": "reference", "metric": "paths/s", "value": value, "unit": "paths/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_s / max(1, len(vals)), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": value / README_BOOK1_10T_PATHS_PER_S if name == "book1_final" else None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": name, "description": wl[8], "note": "CPU restatement of the reference (oracle/, C++ f64, not rustc-built); each step is a bounded sample"},
        "cpu_baseline": {"value": value, "unit": "paths/s", "cores": threads, "kind": "port", "sample": last["sample"]},
        "e2e": {"value": value, "unit": "paths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="rtb200", choices=["rtb200", "reference"])
    ap.add_argument("--workload", default="book1_final", choices=sorted(WORKLOADS))
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel (marks the line as a non-headline configuration)")
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--sharding", default="samples", choices=["samples", "tiles"],
                    help="N>1: sample ranges of every pixel (default) or 4-row tile bands dealt round-robin (SURVEY 8e alternative)")
    ap.add_argument("--reduce", default="peer", choices=["peer", "reduce", "allreduce"],
                    help="N>1: how the accumulators are summed: peer = the library's own kernel over NVLink peer memory (CUDA IPC, rt_peer_*; default), "
                         "reduce / allreduce = one NCCL collective")
    ap.add_argument("--slots", type=int, default=0, help="resident path slots of the wavefront (0 = library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary workloads reported under 'also'")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--frames", type=int, default=0, help="bouncing_anim: number of frames (default 240)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned to its caller as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl rtb200: the reference arm sizes each step's sample from a timing, so its outputs differ from run to run")

    wl = list(WORKLOADS[args.workload])
    if args.spp:
        wl[5] = args.spp
    wl = tuple(wl)
    if args.impl == "reference":
        return reference_arm(args, wl, args.workload)

    import numpy as np
    import torch
    import torch.distributed as dist
    import ray_tracing_series_rust_b200 as rtb
    from ray_tracing_series_rust_b200 import capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: librtb200 has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    api = rtb.load()
    api.lib.rt_scene_set_tuning.restype = C.c_int32

    if args.workload == "bouncing_anim":
        return run_animation(args, wl, api, rtb, capi, torch, dist, world, rank, local)

    sid, sseed, param, W, aspect, spp, depth, cam, desc = wl
    scene = build_scene(rtb, rtb.new_scene, wl)
    t0 = time.time()
    scene.commit()
    commit_s = time.time() - t0
    if args.slots:
        api.lib.rt_scene_set_tuning(C.c_void_p(scene.h), args.slots)
    H = scene.image_height(capi.make_config(W, aspect, 1, depth))

    # sample-range shard of this rank
    from ray_tracing_series_rust_b200 import sharding
    spp_total, s_begin, s_end = sharding.sample_range(spp, rank, world, args.scaling)
    shard_flags = 0
    if args.sharding == "tiles" and world > 1:  # every rank renders all samples of its own bands; weak scaling still grows spp with N
        s_begin, s_end = 0, spp_total
        shard_flags = sharding.tile_flags(rank, world)
    paths_all = W * H * spp_total
    # strong scaling with sample sharding: split the PATHS evenly (rt_render_device_paths), not the samples: 500 spp on 8 GPUs is 62.5 each
    path_shard = None
    if world > 1 and args.scaling == "strong" and not shard_flags:
        path_shard = sharding.path_range(W * H, spp_total, rank, world)
        s_begin, s_end = 0, spp_total

    stream = torch.cuda.current_stream()
    pg = None
    if world > 1 and args.reduce == "peer":
        try:
            pg = sharding.PeerGroup(api, rank, world, W * H * 3)
        except Exception as e:  # no IPC / peer route on this box: the NCCL reduce does the same sum
            print(f"[bench] rank {rank}: peer group unavailable ({e})", file=sys.stderr)
            pg = None
        ok = torch.tensor([1 if pg is not None else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)  # every rank takes the same path
        if int(ok.item()) == 0:
            if pg is not None:
                pg.close()
            pg, args.reduce = None, "reduce"
    accum = torch.zeros((H, W, 3), dtype=torch.int64, device="cuda")
    screen = torch.zeros((H, W, 3), dtype=torch.float64, device="cuda")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    host_screen = torch.empty((H, W, 3), dtype=torch.float64).pin_memory()

    def one_step(step, timed_extend=False, count=False, local_only=False, no_wait=False):
        # no_wait (RT_RENDER_NO_WAIT): the call returns once the render is enqueued, so the reduce and the resolve queue up behind the kernel
        # on the same stream without a host round trip in between (single-launch modes; the wavefront ignores it)
        cfg = capi.make_config(W, aspect, spp_total, depth, seed=1 + step, sample_begin=s_begin, sample_end=s_end,
                               flags=(1 if timed_extend else 0) | (2 if count else 0) | (32 if no_wait else 0) | shard_flags)
        st = capi.Stats()
        sp = C.c_void_p(stream.cuda_stream)
        if pg is not None and not local_only:
            # the library's own exchange: render into the IPC-shared accumulator, publish a flag behind the kernel; rank 0's gather kernel
            # waits for the flags on the device, reads the peers' sums over NVLink and resolves - nothing returns to the host in between
            pg.begin(sp)
            if path_shard is not None:  # an even split of any sample count: whole samples plus a partial first / last one
                api.check(api.render_device_paths(scene.h, C.byref(cfg), path_shard[0], path_shard[1], C.c_void_p(pg.accum), sp, C.byref(st)))
            else:
                api.check(api.render_device(scene.h, C.byref(cfg), C.c_void_p(pg.accum), sp, C.byref(st)))
            pg.publish(sp)
            if rank == 0:
                pg.gather_resolve(C.c_void_p(screen.data_ptr()), W, H, spp_total, H, sp)
            return st.as_dict()
        accum.zero_()
        if path_shard is not None and not local_only:
            api.check(api.render_device_paths(scene.h, C.byref(cfg), path_shard[0], path_shard[1], C.c_void_p(accum.data_ptr()), sp, C.byref(st)))
        else:
            api.check(api.render_device(scene.h, C.byref(cfg), C.c_void_p(accum.data_ptr()), sp, C.byref(st)))
        if local_only:  # rank-0-only diagnostics after the other ranks have left: no collective
            return st.as_dict()
        sharding.reduce_accumulators(accum, dst=0, how=args.reduce)
        if rank == 0:
            api.check(api.resolve_device(C.c_void_p(accum.data_ptr()), C.c_void_p(screen.data_ptr()), W, H, spp_total, H, sp))
        return st.as_dict()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    st_warm = None
    for i in range(args.warmup):
        st_warm = one_step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches = 0
    segments = 0
    paths_local = 0
    t_wall0 = time.time()
    for k in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (outside the timed events)
        barrier()
        ev[k][0].record(stream)
        st = one_step(args.warmup + k, no_wait=True)
        ev[k][1].record(stream)
        launches += st["kernel_launches"] + ((2 + (2 if rank == 0 else 0)) if pg is not None else (1 if rank == 0 else 0))  # flag wait / publish kernels, gather + consumed flag
        if st["segments"] == 0 and st_warm is not None:  # enqueued without waiting: the device counters were not read back; the warm-up render of the same workload has them
            st = st_warm
        segments += st["segments"]
        paths_local += st["paths"]
    barrier()
    t_wall = time.time() - t_wall0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        outs = {"screen": screen.cpu().numpy()}
        if pg is None:  # rank 0 holds the summed accumulator (with the peer group it holds only its own shard)
            outs["accum"] = accum.cpu().numpy().astype(np.float64)
        dump_outputs(args.dump_outputs, outs)
    ms_steps = [a.elapsed_time(b) for a, b in ev]
    ms_local = torch.tensor([sum(ms_steps)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms_local, op=dist.ReduceOp.MAX)
    ms_total = float(ms_local.item())
    ms_per_step = ms_total / args.steps
    value = paths_all * args.steps / (ms_total * 1e-3)

    if os.environ.get("RTB200_BENCH_DEBUG"):  # per-rank device time of this rank's shard alone (waits for the kernel: not part of any reported number)
        barrier()
        ms_dbg = []
        for k in range(3):
            flush.zero_()
            barrier()
            ms_dbg.append(one_step(2000 + k, local_only=True)["ms_device"])
        print(f"[bench debug] rank {rank}: shard spp {s_end - s_begin}, k_mega ms {[round(x, 3) for x in ms_dbg]}, ideal {ms_per_step:.3f} step", file=sys.stderr, flush=True)
        barrier()
    if pg is not None:
        torch.cuda.synchronize()
        if pg.timed_out():
            raise SystemExit("bench.py: a peer never published its accumulator (rt_peer_timed_out)")
    # ---- book-2 final, the other north-star render, split the same way (all ranks; one timed render after a short warm-up)
    book2 = None
    if not args.no_extra and args.workload == "book1_final" and not args.spp and args.scaling == "strong":
        book2 = strong_render(api, rtb, capi, sharding, torch, dist, stream, "book2_final", rank, world, barrier)

    out_hc = (C.c_int64 * 16)()
    api.lib.rt_scene_host_check.restype = C.c_int32
    api.lib.rt_scene_host_check(C.c_void_p(scene.h), out_hc)
    scene_bytes = int(out_hc[14])

    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()  # every collective is done; rank 0 continues alone (e2e, roofline, CPU baseline)
    if rank != 0:
        return 0

    # ---- e2e: the plugin call with HOST buffers, as a Rust render_scene_gpu would make it (world.rs:1181 seam), rank 0 alone:
    # rt_scene_commit[_multi] (flatten + BVH + H2D of the scene to every GPU) + rt_render[_multi] (kernels on all N GPUs, peer-memory
    # reduce + resolve, D2H of the Screen into a pageable numpy buffer), wall clock around the calls, same spp as the timed steps
    n_dev = torch.cuda.device_count()
    e2e_gpus = world if n_dev >= world else 1
    e2e_ms, e2e_commit_ms = [], []
    cfg_e = capi.make_config(W, aspect, spp_total, depth, seed=100)
    for k in range(args.warmup + args.steps):
        cfg_e.seed = 100 + k
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if e2e_gpus > 1:
            scene.commit_multi(e2e_gpus)
            t1 = time.perf_counter()
            scr_e, _, st_e = scene.render_multi(cfg_e, e2e_gpus, capi.RT_SHARD_SAMPLES)
        else:
            scene.commit()
            t1 = time.perf_counter()
            scr_e, _, st_e = scene.render(cfg_e)
        t2 = time.perf_counter()
        if k >= args.warmup:
            e2e_ms.append(1e3 * (t2 - t0))
            e2e_commit_ms.append(1e3 * (t1 - t0))
            launches_e2e = st_e["kernel_launches"] + 1
    e2e_ms_avg = sum(e2e_ms) / len(e2e_ms)
    e2e_value = W * H * spp_total / (e2e_ms_avg * 1e-3)

    # ---- roofline of the dominant kernel, rank 0.  RT_MODE_AUTO picks the fused persistent kernel (k_mega: one launch
    # per render, path state in registers) or the wavefront (k_extend dominant: CUDA events around every launch).
    st_n = one_step(1000, local_only=True)
    fused = st_n["iterations"] == 1
    st_c = one_step(1000, count=True, local_only=True)  # device event counters (runs the wavefront; same rays, same BVH work)
    if fused:
        n_ext = 1
        ext_ms_avg = st_n["ms_device"]
        seg_per_launch = float(st_n["segments"])
        ext_share = 1.0
    else:
        st_t = one_step(1000, timed_extend=True, local_only=True)
        n_ext = max(1, st_t["iterations"])
        ext_ms_avg = st_t["ms_extend"] / n_ext
        seg_per_launch = st_t["segments"] / n_ext
        ext_share = st_t["ms_extend"] / max(st_t["ms_device"], 1e-9)
    hbm, hbm_src = peaks()

    cpu = None
    algo = None
    if not args.no_cpu_baseline and world == 1:  # the CPU baseline is reported at N=1 only (the other ranks have left; keep the N>1 lines short)
        c = run_cpu_sample(wl, args.cpu_seconds, os.cpu_count() or 1)
        algo = oracle_counts_per_segment(c["stats"])
        cpu = {"value": c["paths_per_s"], "unit": "paths/s", "cores": os.cpu_count() or 1, "kind": "port", "sample": c["sample"],
               "segments_per_path": algo["segments_per_path"]}
    # Algorithmic bytes per segment (SURVEY.md 8d): 32 B per BVH box tested + per-primitive bytes + 160 B of
    # wavefront path state.  The box / primitive counts are the kernel's OWN (device counters on the same
    # workload): the reference's median-split x/y BVH tests ~2.5x more boxes per ray than the SAH tree this
    # kernel walks, so crediting the kernel with the reference's counts would overstate it.  The
    # reference-count variant is reported next to it as `reference_counts`.
    own_seg = max(st_c["segments"], 1)
    prim_b = B_PRIM[{13: 0, 99: 1, 5: 4, 6: 4, 14: 5}.get(sid, 0)]
    state_b = 0 if fused else B_STATE  # the fused kernel keeps the path state in registers: no state traffic to count
    own_bps = B_NODE * st_c["box_tests"] / own_seg + prim_b * st_c["prim_tests"][0] / own_seg + state_b
    achieved = own_bps * seg_per_launch / (ext_ms_avg * 1e-3) / 1e9
    roofline = {
        # What binds is SIMT issue (divergent incoherent rays), not DRAM: the scene is L1/L2 resident (`traffic` is a few 1e-5 of the
        # algorithmic bytes).  achieved / peak / frac stay the SURVEY 8(d) HBM figure (algorithmic bytes over measured copy bandwidth);
        # `frac_binding` = lane-issue efficiency of the same kernel from the committed ncu capture (issue-active x active threads / 32).
        "bound": "issue", "kernel": "k_mega (fused persistent: generate + world.hit + scatter)" if fused else "k_extend",
        "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "traffic": None,
        "peak_source": hbm_src,
        "bytes_per_segment": own_bps,
        "bytes_per_segment_source": "device event counters: BVH boxes tested x 32 B + primitive tests x B_type" + ("" if fused else " + 160 B wavefront state"),
        "nodes_per_segment": st_c["box_tests"] / own_seg, "prim_tests_per_segment": st_c["prim_tests"][0] / own_seg,
        "segments_per_launch": seg_per_launch, "launch_ms_avg": ext_ms_avg, "launches_timed": n_ext,
        "kernel_share_of_step": ext_share,
        "note": "the scene (<64 KB) is L1/L2 resident, so DRAM traffic is far below the algorithmic bytes; the kernel is issue/latency bound, see profiles/",
    }
    try:
        wide = fused and scene.bvh_width() == 4
    except Exception:
        wide = False
    if wide:
        # the counting pass walks the same 4-wide collapse as the timed fused kernel (kernels.cu count_wide): box_tests = 4 per node
        # visited, so 32 B x box_tests = 128 B per visit = the bytes of the nodes the kernel fetches
        roofline["kernel"] = ("k_mega" if sid == 13 else "k_mega_r (resumable)") + " (fused persistent: generate + world.hit + scatter; 4-wide BVH walk)"
        roofline["bytes_per_segment_source"] = "device event counters on the 4-wide tree the kernel walks: node visits x 128 B (= boxes tested x 32 B) + primitive tests x B_type"
        roofline["wide_node_visits_per_segment"] = st_c["box_tests"] / own_seg / 4.0
    if fused and sid == 99:
        roofline["note"] += "; the box / primitive counts come from the counting wavefront pass, which walks union-over-the-shutter boxes: the fused kernel walks motion-interpolated boxes and tests fewer, so `achieved` is an upper bound for this workload"
    if algo:
        ref_ach = (algo["bytes_per_segment"] - (B_STATE if fused else 0)) * seg_per_launch / (ext_ms_avg * 1e-3) / 1e9
        roofline["reference_counts"] = {"bytes_per_segment": algo["bytes_per_segment"] - (B_STATE if fused else 0), "box_tests_per_segment": algo["box_tests_per_segment"],
                                        "prim_tests_per_segment": algo["prim_tests_per_segment"], "achieved": ref_ach, "frac": ref_ach / hbm}
    # second ceiling (SURVEY.md 8d): FP32 issue, nominal 148 SMs x 128 lanes x 2 x SM clock; flops per segment from the same
    # device counters with the survey's per-test constants (box 20, sphere 30, moving sphere 40, rect 12, triangle 70, shading ~90)
    f_prim = {13: 30, 99: 40, 5: 12, 6: 30, 14: 70}.get(sid, 30)
    fps = 20.0 * st_c["box_tests"] / own_seg + f_prim * st_c["prim_tests"][0] / own_seg + 90.0
    fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12
    fl_ach = fps * seg_per_launch / (ext_ms_avg * 1e-3) / 1e12
    roofline["second_ceiling"] = {"kind": "fp32 issue, nominal (148 SM x 128 lanes x 2 x 1.965 GHz)", "flops_per_segment": fps, "achieved": fl_ach,
                                  "peak": fp32_peak, "unit": "TFLOP/s", "frac": fl_ach / fp32_peak}
    prof = os.path.join(ROOT, "profiles", "extend_traffic.json")
    if os.path.exists(prof):
        try:
            pj = json.load(open(prof)).get(args.workload, {}).get("fused" if fused else "wavefront", {})
            roofline["traffic"] = pj.get("dram_bytes_per_launch")
            roofline["traffic_source"] = f"profiles/extend_traffic.json (ncu --set full capture {pj.get('capture', '?')}, kernel {pj.get('kernel', '?')}); not re-measured by this run"
            if "ncu" in pj:
                roofline["ncu"] = pj["ncu"]  # issue-slot utilisation, active threads per instruction, stalls: what actually bounds the kernel
                ia, th = pj["ncu"].get("issue_active_pct"), pj["ncu"].get("threads_per_instruction")
                if ia and th:
                    roofline["frac_binding"] = (ia / 100.0) * (th / 32.0)
                    roofline["binding"] = {"roof": "SIMT lane-issue slots (4 schedulers x 32 lanes per SM per cycle)", "issue_active": ia / 100.0, "active_threads_per_instruction": th,
                                           "frac": (ia / 100.0) * (th / 32.0)}
        except Exception:
            pass

    line = {
        "metric": "paths/s", "value": value, "unit": "paths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": (value / README_BOOK1_10T_PATHS_PER_S) if (args.workload == "book1_final" and not args.spp) else None,
        "dtype": "f64 geometry / f32 slabs+colour", "data": "synthetic",
        "config": {"workload": args.workload, "description": desc, "image": [W, H], "spp_per_gpu": (spp_total / world) if path_shard is not None else (s_end - s_begin), "spp_total": spp_total, "max_depth": depth,
                   "paths_per_step": paths_all, "segments_per_path": segments / max(1, paths_local),
                   "sharding": ("single GPU" if world == 1 else (("4-row tile bands round-robin" if shard_flags else "sample ranges") +
                                                                      (" + the library's peer-memory gather (CUDA IPC, k_reduce_resolve on rank 0 reads the shards over NVLink)" if pg is not None
                                                                       else f" + one NCCL int64 {args.reduce} to rank 0"))),
                   "render_mode": "fused persistent kernel (RT_MODE_AUTO)" if fused else "wavefront (RT_MODE_AUTO)",
                   "l2": "flushed between timed steps (256 MiB memset, untimed); path state > L2",
                   "vs_baseline_note": "README.md:23 146.440 s on 10 threads of an unspecified CPU => 1.456e6 paths/s (derived)",
                   "render_wall_s": ms_per_step * 1e-3, "commit_s": commit_s, "wall_s_timed_region": t_wall},
        "e2e": {"value": e2e_value, "unit": "paths/s", "h2d_bytes_per_step": scene_bytes * e2e_gpus, "d2h_bytes_per_step": W * H * 3,
                "ms_per_step": e2e_ms_avg, "commit_ms": sum(e2e_commit_ms) / len(e2e_commit_ms), "steps": len(e2e_ms), "n_gpus": e2e_gpus,
                "call": ("rt_scene_commit + rt_render" if e2e_gpus == 1 else "rt_scene_commit_multi + rt_render_multi (one process, peer-memory reduce + resolve)") +
                        " with a host f64 Screen buffer (numpy, pageable); wall clock around the two calls",
                "d2h_note": "the Screen crosses PCIe as bytes (every value is an integer 0..255) and is widened to the reference's f64 Colors on the host",
                "gpu_launches_per_step": int(launches_e2e)},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu,
    }
    if not args.no_extra and world == 1 and args.workload == "book1_final" and not args.spp:
        line["also"] = extra_workloads(api, rtb, capi, stream, args)
    if book2 is not None:
        line.setdefault("also", {})["book2_final_strong"] = book2
    print(json.dumps(line), flush=True)
    return 0


def strong_render(api, rtb, capi, sharding, torch, dist, stream, name, rank, world, barrier):
    """One full render of WORKLOADS[name] split into `world` sample ranges (strong scaling), timed on the device (max over ranks):
    render_device + NCCL reduce + resolve.  Returns the record on rank 0, None elsewhere."""
    sid, sseed, param, W, aspect, spp, depth, cam, desc = WORKLOADS[name]
    s = rtb.new_scene()
    s.world_build(sid, sseed, param)
    s.commit()
    H = s.image_height(capi.make_config(W, aspect, 1, depth))
    accum = torch.zeros((H, W, 3), dtype=torch.int64, device="cuda")
    screen = torch.zeros((H, W, 3), dtype=torch.float64, device="cuda")

    def render(total, seed):
        _, b, e = sharding.sample_range(total, rank, world, "strong")
        cfg = capi.make_config(W, aspect, total, depth, seed=seed, sample_begin=b, sample_end=e)
        accum.zero_()
        st = capi.Stats()
        if e > b:
            api.check(api.render_device(s.h, C.byref(cfg), C.c_void_p(accum.data_ptr()), C.c_void_p(stream.cuda_stream), C.byref(st)))
        sharding.reduce_accumulators(accum, dst=0)
        if rank == 0:
            api.check(api.resolve_device(C.c_void_p(accum.data_ptr()), C.c_void_p(screen.data_ptr()), W, H, total, H, C.c_void_p(stream.cuda_stream)))
        return st.as_dict()
    render(8 * world, 1)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(stream)
    st = render(spp, 3)
    e1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    seg = torch.tensor([float(st["segments"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(seg, op=dist.ReduceOp.SUM)
    s.close()
    if rank != 0:
        return None
    t = float(ms.item()) * 1e-3
    return {"description": desc, "n_gpus": world, "scaling": "strong", "spp_total": spp, "spp_per_gpu": spp / world, "paths": W * H * spp,
            "render_wall_s": t, "host_wall_s": wall, "paths_per_s": W * H * spp / t, "segments_per_path": float(seg.item()) / (W * H * spp),
            "timing": "CUDA events around render_device + NCCL int64 reduce + resolve, max over ranks; one full render after an 8-spp-per-GPU warm-up"}


def run_animation(args, wl, api, rtb, capi, torch, dist, world, rank, local):
    """BASELINE configs[4]: frame f -> rank f mod world, no collective.  A step renders every frame once:
    rt_scene_set_camera(shutter) + rt_scene_commit (GravitySphere windows, BVH) + render + resolve + D2H."""
    from ray_tracing_series_rust_b200 import sharding
    sid, sseed, n_frames, W, aspect, spp, depth, cam, desc = wl
    if args.frames:
        n_frames = args.frames
    scene = rtb.new_scene()
    scene.world_build(sid, sseed, 0)
    cfg0 = capi.make_config(W, aspect, spp, depth)
    H = scene.image_height(cfg0)
    stream = torch.cuda.current_stream()
    accum = torch.zeros((H, W, 3), dtype=torch.int64, device="cuda")
    screen = torch.zeros((H, W, 3), dtype=torch.float64, device="cuda")
    host = torch.empty((H, W, 3), dtype=torch.float64).pin_memory()
    mine = sharding.frames_for_rank(n_frames, rank, world)
    dump_frames = []
    if args.dump_outputs and rank == 0 and mine:  # 240 Screens are 2.5 GB: keep 8 evenly spaced ones (8 x 5.1 MB as float32)
        dump_frames = [mine[i] for i in sorted({round(j * (len(mine) - 1) / 7) for j in range(8)})]

    def step(k, keep=None):
        launches = 0
        for f in mine:
            scene.set_camera((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, aspect, 0.1, 10.0, 0.4 * f, 0.4 * f + 0.4)
            scene.commit()
            cfg = capi.make_config(W, aspect, spp, depth, seed=5 + f + 1000 * k)
            accum.zero_()
            st = capi.Stats()
            api.check(api.render_device(scene.h, C.byref(cfg), C.c_void_p(accum.data_ptr()), C.c_void_p(stream.cuda_stream), C.byref(st)))
            api.check(api.resolve_device(C.c_void_p(accum.data_ptr()), C.c_void_p(screen.data_ptr()), W, H, spp, H, C.c_void_p(stream.cuda_stream)))
            host.copy_(screen, non_blocking=True)
            if keep is not None and f in dump_frames:
                keep[f] = screen.float()  # a device copy on the same stream: the next frame overwrites `screen`
            launches += st.kernel_launches + 1
        torch.cuda.synchronize()
        return launches

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    t0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    launches = 0
    kept = {} if dump_frames else None
    for k in range(args.steps):
        launches += step(args.warmup + k, kept if k == args.steps - 1 else None)
    e1.record(stream)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if kept:
        dump_outputs(args.dump_outputs, {"screen_frame%03d" % f: kept[f].cpu().numpy() for f in dump_frames})
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0
    ms_total = float(ms.item())
    paths_step = W * H * spp * n_frames
    value = paths_step * args.steps / (ms_total * 1e-3)
    line = {"metric": "paths/s", "value": value, "unit": "paths/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "bouncing_anim", "description": desc, "frames": n_frames, "image": [W, H], "spp": spp, "max_depth": depth,
                       "sharding": "frame f -> rank f mod N, no collective", "frames_per_s": n_frames * args.steps / (ms_total * 1e-3),
                       "l2": "every frame re-commits the scene and streams > L2 of path state", "wall_s": time.time() - t0},
            "e2e": {"value": value, "unit": "paths/s", "h2d_bytes_per_step": None, "d2h_bytes_per_step": W * H * 3 * 8 * n_frames,
                    "note": "the timed region already contains per-frame commit (H2D) and Screen D2H: value == e2e"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": None, "cpu_baseline": None}
    print(json.dumps(line), flush=True)
    return 0


def extra_workloads(api, rtb, capi, stream, args=None):
    """One timed render each of the other BASELINE configs (single GPU), so every headline config has a
    measured paths/s in the round's bench record.  book2_final runs its full 10 000 spp only when a
    100-spp probe projects under 100 s; otherwise the probe is reported and flagged."""
    import torch
    out = {}
    try:  # BASELINE configs[4]: 6 frames of the 240-frame animation, per-frame commit included
        sid, sseed, n_frames, W, aspect, spp, depth, cam, desc = WORKLOADS["bouncing_anim"]
        s = rtb.new_scene()
        s.world_build(sid, sseed, 0)
        H = s.image_height(capi.make_config(W, aspect, 1, depth))
        accum = torch.zeros((H, W, 3), dtype=torch.int64, device="cuda")
        t_frames, paths = 0.0, 0
        for i, f in enumerate((0, 0, 40, 80, 120, 160, 200)):
            torch.cuda.synchronize()
            t0 = time.time()
            s.set_camera((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, aspect, 0.1, 10.0, 0.4 * f, 0.4 * f + 0.4)
            s.commit()
            accum.zero_()
            st = capi.Stats()
            api.check(api.render_device(s.h, C.byref(capi.make_config(W, aspect, spp, depth, seed=5 + f)), C.c_void_p(accum.data_ptr()), C.c_void_p(stream.cuda_stream), C.byref(st)))
            torch.cuda.synchronize()
            if i > 0:
                t_frames += time.time() - t0
                paths += st.paths
        out["bouncing_anim"] = {"description": desc, "frames_timed": 6, "paths_per_s": paths / t_frames, "s_per_frame": t_frames / 6,
                                "projected_240_frames_wall_s": 240 * t_frames / 6, "includes": "per-frame set_camera + commit + render"}
        s.close()
        del accum
    except Exception as e:
        out["bouncing_anim"] = {"error": str(e)}
    for name in ("book1_shipped", "cornell_smoke", "mesh_room"):  # book2_final: see also.book2_final_strong (the full 10 000 spp)
        sid, sseed, param, W, aspect, spp, depth, cam, desc = WORKLOADS[name]
        try:
            s = rtb.new_scene()
            t0 = time.time()
            s.world_build(sid, sseed, param)
            build_s = time.time() - t0
            t0 = time.time()
            s.commit()
            commit_s = time.time() - t0
            H = s.image_height(capi.make_config(W, aspect, 1, depth))
            accum = torch.zeros((H, W, 3), dtype=torch.int64, device="cuda")

            def render(n_spp, total):
                cfg = capi.make_config(W, aspect, total, depth, seed=7, sample_begin=0, sample_end=n_spp)
                accum.zero_()
                st = capi.Stats()
                api.check(api.render_device(s.h, C.byref(cfg), C.c_void_p(accum.data_ptr()), C.c_void_p(stream.cuda_stream), C.byref(st)))
                torch.cuda.synchronize()
                return st.as_dict()
            probe_spp = min(spp, 100 if name != "mesh_room" else 20)
            render(min(4, spp), spp)
            st = render(probe_spp, spp)
            rate = st["paths"] / (st["ms_device"] * 1e-3)
            full_s = W * H * spp / rate
            rec = {"description": desc, "build_s": build_s, "commit_s": commit_s}
            if full_s <= 100.0 and probe_spp < spp:
                st = render(spp, spp)
                rec.update({"spp": spp, "full_config": True})
            else:
                rec.update({"spp": probe_spp, "full_config": probe_spp == spp, "projected_full_wall_s": full_s})
            rec.update({"paths_per_s": st["paths"] / (st["ms_device"] * 1e-3), "render_wall_s": st["ms_device"] * 1e-3,
                        "segments_per_path": st["segments"] / max(1, st["paths"]), "iterations": st["iterations"]})
            out[name] = rec
            s.close()
            del accum
        except Exception as e:  # a secondary workload must not take the headline line down
            out[name] = {"error": str(e)}
    if args is not None and not args.no_cpu_baseline:
        # BASELINE.md section 2: the CPU restatement of the reference beside every config, all host cores, on a BOUNDED sample of each
        # (full image at a reduced spp; paths/s does not depend on spp, so the full-config wall time is a linear extrapolation: flagged)
        cpus = {}
        per = max(3.0, min(8.0, args.cpu_seconds / 2))
        for name in ("cornell_smoke", "book2_final", "mesh_room", "bouncing_anim"):
            try:
                wl = WORKLOADS[name]
                if name == "mesh_room":
                    # the reference builds its BVH by cloning the object list per node (bvh.rs:14-83): minutes for 871 200 triangles, so the
                    # CPU sample uses the same room around a 131 072-triangle mesh (param 256) - per-path cost grows with log(triangles): optimistic for the CPU
                    wl = wl[:2] + (256,) + wl[3:]
                if name == "bouncing_anim":
                    wl = wl[:2] + (0,) + wl[3:]  # one frame of the animation scene (param = frame count is a bench notion, not a scene size)
                c = run_cpu_sample(wl, per, os.cpu_count() or 1, width=wl[3] // 4)  # a quarter of the width: the 1-spp calibration pass stays short
                W, aspect, spp = wl[3], wl[4], wl[5]
                full_paths = c["stats"]["paths"] / c["spp"] * 16.0 * spp * (WORKLOADS[name][2] if name == "bouncing_anim" else 1)
                cpus[name] = {"value": c["paths_per_s"], "unit": "paths/s", "cores": os.cpu_count() or 1, "kind": "port", "sample": c["sample"],
                              "extrapolated_full_config_wall_s": full_paths / c["paths_per_s"], "extrapolated": True,
                              "note": ("131 072-triangle stand-in mesh (see bench.py)" if name == "mesh_room" else
                                       ("one frame (shutter [0, 10)), extrapolated to 240 frames; CPU commit / table integration not included" if name == "bouncing_anim" else ""))}
            except Exception as e:
                cpus[name] = {"error": str(e)}
        out["cpu_baselines"] = cpus
    try:  # SURVEY.md 8(f) n1 / n2 on the mesh-room inputs: commit with the host SAH vs the device LBVH builder, text vs binary I/O
        import glob
        import numpy as np
        sid, sseed, param, W, aspect, spp, depth, cam, desc = WORKLOADS["mesh_room"]
        rec = {}
        for label, builder in (("host_sah", 0), ("device_lbvh", 1)):
            for attempt in ("first", "warm"):  # the first device build also pays CUDA's lazy loading of the sort / scan kernels
                s = rtb.new_scene()
                s.world_build(sid, sseed, param)
                s.set_bvh_builder(builder)
                t0 = time.time()
                s.commit()
                rec[label + ("_commit_first_s" if attempt == "first" else "_commit_s")] = time.time() - t0
                if attempt == "first":
                    s.close()
            rec[label + "_device_built_prims"] = s.host_check()["device_built_prims"] if builder else 0
            cfg = capi.make_config(W, aspect, 20, depth, seed=7)
            s.render(cfg)
            st = s.render(cfg)[2]
            rec[label + "_paths_per_s"] = st["paths"] / (st["ms_device"] * 1e-3)
            s.close()
        plys = sorted(glob.glob("/tmp/rtb200_mesh_*_%d.ply" % param))  # the mesh world_build(14) wrote (world.hpp stanford_dragon)
        with tempfile.TemporaryDirectory(prefix="rtb200_bench_") as tmp:  # the files written here never go under the source tree
            if plys:
                binp = os.path.join(tmp, "mesh.bin.ply")
                capi.ply_convert_binary(api, plys[-1], binp)
                for label, path in (("ply_ascii", plys[-1]), ("ply_binary", binp)):
                    s = rtb.new_scene()
                    m = s.lambertian((0.2, 0.2, 0.2))
                    t0 = time.time()
                    s.ply_load(path, 1.0, m)
                    rec[label + "_load_s"] = time.time() - t0
                    rec[label + "_MB"] = os.path.getsize(path) / 1e6
                    s.close()
            scr = np.random.default_rng(0).integers(0, 256, size=(1000, 1000, 3)).astype(np.float64)
            outp = os.path.join(tmp, "io.ppm")
            for label, fn in (("ppm_p3", capi.write_ppm), ("ppm_p6", capi.write_ppm_binary)):
                t0 = time.time()
                fn(api, outp, scr)
                rec[label + "_write_s"] = time.time() - t0
        out["next_rows"] = {"description": "SURVEY 8(f): n1 commit of the 871200-triangle mesh room per BVH builder (+ paths/s of the tree at 20 spp); "
                                           "n2 ASCII vs binary PLY load of that mesh, P3 vs P6 write of a 1000x1000 Screen (host)", **rec}
    except Exception as e:
        out["next_rows"] = {"error": str(e)}
    return out


if __name__ == "__main__":
    sys.exit(main())
