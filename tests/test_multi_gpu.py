"""rt_render_multi — multi-GPU inside the C-ABI (SURVEY.md 8(b) n_gpus / shard_mode, 8(e); seam: render_scene, world.rs:1181-1247,
whose row-band fan-out + mpsc gather, world.rs:1198-1240, this replaces).

One process renders one shard per GPU and one kernel on GPU 0 sums the shards' int64 accumulators where they lie (peer memory)
and resolves the Screen.  Bars: the image and the accumulator are BIT-IDENTICAL to the single-GPU rt_render for every GPU count
and both shard modes, in both render modes.  On a 1-GPU box RTB200_MULTI_ALIAS=1 maps every logical GPU onto the one device
(separate scene arenas, accumulators, streams, workspaces): the whole host logic and the reduce + resolve kernel run; with two
or more devices visible the test also runs over real peers."""
import os

import numpy as np
import pytest

import ray_tracing_series_rust_b200 as rtb
from ray_tracing_series_rust_b200 import capi


def _device_count():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


@pytest.fixture
def alias(monkeypatch):
    monkeypatch.setenv("RTB200_MULTI_ALIAS", "1")


def _scene(scene_id, seed=0xB001, param=0):
    g = rtb.new_scene()
    g.world_build(scene_id, seed, param)
    g.commit()
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,width,aspect", [(13, 96, 1.5), (5, 64, 1.0), (14, 64, 1.0)])
def test_multi_is_bit_identical_to_single(alias, scene_id, width, aspect):
    """fused (13, 14) and wavefront (5: media) scenes; 2 / 3 / 8 shards; sample ranges and tile bands; spp not divisible by 3 or 8"""
    g = _scene(scene_id, param=40 if scene_id == 14 else 0)
    cfg = capi.make_config(width, aspect, 7, 50, seed=21, compat_threads=5)
    s1, a1, st1 = g.render(cfg, want_accum=True)
    assert a1.any() and (s1[-1] == 0).all()  # compat_threads: the top rows stay black on every path
    for n in (2, 3, 8):
        for mode in (capi.RT_SHARD_SAMPLES, capi.RT_SHARD_TILES):
            sn, an, stn = g.render_multi(cfg, n, mode, want_accum=True)
            assert np.array_equal(an, a1) and np.array_equal(sn, s1), (scene_id, n, mode)
            assert stn["paths"] == st1["paths"] and stn["segments"] == st1["segments"]
    # screen only (no accumulator requested) and a sub-range of the samples
    sn, an, _ = g.render_multi(cfg, 4, capi.RT_SHARD_SAMPLES)
    assert an is None and np.array_equal(sn, s1)
    sub = capi.make_config(width, aspect, 7, 50, seed=21, compat_threads=5, sample_begin=2, sample_end=7)
    _, a_sub1, _ = g.render(sub, want_accum=True)
    _, a_subn, _ = g.render_multi(sub, 3, capi.RT_SHARD_SAMPLES, want_accum=True)
    assert np.array_equal(a_sub1, a_subn)
    g.close()


@pytest.mark.gpu
def test_multi_follows_recommits_and_background_changes(alias):
    """replicas re-upload after a commit (new camera shutter -> new bounds) and track scalar changes made after it"""
    g = _scene(8, seed=0xB005)
    cfg = capi.make_config(80, 1.5, 4, 50, seed=4)
    for f in (0, 30):
        g.set_camera((13, 2, 3), (0, 0, 0), (0, 1, 0), 20.0, 1.5, 0.1, 10.0, 0.4 * f, 0.4 * f + 0.4)
        g.commit_multi(2) if f == 0 else g.commit()
        _, a1, _ = g.render(cfg, want_accum=True)
        _, a2, _ = g.render_multi(cfg, 2, capi.RT_SHARD_TILES, want_accum=True)
        assert np.array_equal(a1, a2), f
    g.set_background((0.1, 0.2, 0.9))
    _, a1, _ = g.render(cfg, want_accum=True)
    _, a2, _ = g.render_multi(cfg, 2, want_accum=True)
    assert np.array_equal(a1, a2)
    g.close()


@pytest.mark.gpu
def test_multi_argument_errors(monkeypatch):
    monkeypatch.delenv("RTB200_MULTI_ALIAS", raising=False)
    g = _scene(13)
    cfg = capi.make_config(32, 1.5, 2, 5)
    with pytest.raises(capi.RtError) as e:
        g.render_multi(cfg, 0)
    assert e.value.code == -1
    with pytest.raises(capi.RtError) as e:
        g.render_multi(cfg, 2, 7)
    assert e.value.code == -1
    with pytest.raises(capi.RtError) as e:
        g.render_multi(cfg, _device_count() + 1)  # more GPUs than the box has
    assert e.value.code == -1 and "devices" in str(e.value)
    monkeypatch.setenv("RTB200_MULTI_ALIAS", "1")
    with pytest.raises(capi.RtError) as e:
        g.render_multi(capi.make_config(32, 1.5, 2, 5, flags=(1 << 16) | (2 << 24)), 2)  # RT_RENDER_TILE_SHARD(1, 2): the call shards the image itself
    assert e.value.code == -1
    g.close()


@pytest.mark.gpu
@pytest.mark.skipif(_device_count() < 2, reason="needs two visible GPUs")
def test_multi_over_real_peers():
    """no alias: GPU 0 reads GPU 1..n-1's accumulators over NVLink in k_reduce_resolve"""
    n_dev = _device_count()
    g = _scene(13)
    cfg = capi.make_config(200, 1.5, 16, 50, seed=2)
    s1, a1, _ = g.render(cfg, want_accum=True)
    for n in sorted({2, n_dev}):
        for mode in (capi.RT_SHARD_SAMPLES, capi.RT_SHARD_TILES):
            sn, an, st = g.render_multi(cfg, n, mode, want_accum=True)
            assert np.array_equal(an, a1) and np.array_equal(sn, s1), (n, mode)
    g.close()
    w = _scene(6, seed=0xB002)  # wavefront mode on every GPU (media + Perlin)
    cfgw = capi.make_config(120, 1.0, 6, 50, seed=3)
    _, aw1, _ = w.render(cfgw, want_accum=True)
    _, awn, _ = w.render_multi(cfgw, n_dev, want_accum=True)
    assert np.array_equal(aw1, awn)
    w.close()


def test_multi_symbols_are_exported_and_refuse_without_gpu():
    """CPU box: the entry points exist; without a device they fail like rt_render does (no CPU fallback)"""
    api = rtb.load()
    assert hasattr(api.lib, "rt_render_multi") and hasattr(api.lib, "rt_scene_commit_multi")
    if _device_count() == 0:
        s = rtb.new_scene()
        s.world_build(13, 1)
        with pytest.raises(capi.RtError) as e:
            s.commit_multi(2)
        assert e.value.code == -5
        with pytest.raises(capi.RtError) as e:
            s.render_multi(capi.make_config(32, 1.5, 1, 5), 2)
        assert e.value.code == -2  # not committed


# ---------------------------------------------------------------- peer group: one process per GPU, exchange over CUDA IPC
def _peer_worker(rank, world, port, out_path, n_dev):
    import sys
    import ctypes as C
    import torch
    import torch.distributed as dist
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in sys.path:
        sys.path.insert(0, root)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)  # plumbing only: hands the IPC handles round
    torch.cuda.set_device(rank % n_dev)  # two processes share cuda:0 on a 1-GPU box: CUDA IPC works between processes on one device too
    import ray_tracing_series_rust_b200 as rtb
    from ray_tracing_series_rust_b200 import capi, sharding
    api = rtb.load()
    g = rtb.new_scene()
    g.world_build(13, 0xB001, 0)
    g.commit()
    W, aspect, spp = 120, 1.5, 9
    H = g.image_height(capi.make_config(W, aspect, 1, 50))
    pg = sharding.PeerGroup(api, rank, world, W * H * 3)
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)
    screen = torch.zeros((H, W, 3), dtype=torch.float64, device="cuda")
    outs = []
    for step in range(3):  # several steps: begin() must wait for rank 0's consumption of the previous one
        _, b, e = sharding.sample_range(spp, rank, world, "strong")
        cfg = capi.make_config(W, aspect, spp, 50, seed=40 + step, sample_begin=b, sample_end=e, flags=32)  # RT_RENDER_NO_WAIT
        pg.begin(sp)
        st = capi.Stats()
        api.check(api.render_device(g.h, C.byref(cfg), C.c_void_p(pg.accum), sp, C.byref(st)))
        pg.publish(sp)
        if rank == 0:
            pg.gather_resolve(C.c_void_p(screen.data_ptr()), W, H, spp, H, sp)
            torch.cuda.synchronize()
            outs.append(screen.cpu().numpy().copy())
    torch.cuda.synchronize()
    assert not pg.timed_out()
    dist.barrier()
    if rank == 0:
        np.save(out_path, np.stack(outs))
    pg.close()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_peer_group_gather_equals_single_render(tmp_path):
    """two processes (one GPU each when the box has two, else both on cuda:0) render sample ranges into IPC-shared accumulators;
    rank 0's k_reduce_resolve waits for the published flags, sums the shards where they lie and resolves: the Screen of every
    step equals the single-process rt_render Screen of the same seed, bit for bit"""
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    out = str(tmp_path / "peer_screens.npy")
    world = 2
    mp.spawn(_peer_worker, args=(world, port, out, max(1, _device_count())), nprocs=world, join=True)
    got = np.load(out)
    g = _scene(13)
    for step in range(3):
        ref, _, _ = g.render(capi.make_config(120, 1.5, 9, 50, seed=40 + step))
        assert np.array_equal(got[step], ref), step
    g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scene_id,flags", [(13, 0), (13, 4), (5, 0), (14, 0)])
def test_path_range_shards_add_up(scene_id, flags):
    """rt_render_device_paths: N contiguous ranges of the sample-major path enumeration (whole samples plus partial ones) sum to the
    whole render, bit for bit, for shard counts that do not divide the sample count; fused, wavefront and resumable kernels"""
    import ctypes as C
    import torch
    from ray_tracing_series_rust_b200 import sharding
    api = rtb.load()
    g = _scene(scene_id, param=40 if scene_id == 14 else 0)
    W, aspect, spp = 72, 1.0 if scene_id != 13 else 1.5, 5
    cfg = capi.make_config(W, aspect, spp, 50, seed=8, flags=flags)
    _, ref, st_ref = g.render(cfg, want_accum=True)
    H = ref.shape[0]
    stream = torch.cuda.current_stream()
    for n in (3, 8):
        acc = torch.zeros((H, W, 3), dtype=torch.int64, device="cuda")
        paths = 0
        for r in range(n):
            b, e = sharding.path_range(W * H, spp, r, n)
            st = capi.Stats()
            api.check(api.render_device_paths(g.h, C.byref(cfg), b, e, C.c_void_p(acc.data_ptr()), C.c_void_p(stream.cuda_stream), C.byref(st)))
            paths += st.paths
        torch.cuda.synchronize()
        assert paths == st_ref["paths"] and np.array_equal(acc.cpu().numpy(), ref), (scene_id, n)
    g.close()
