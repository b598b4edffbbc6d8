"""Host logic of the multi-GPU partitioning: frame shards, row bands, and the halo exchange run with
world_size 2 and 3 on CPU (gloo), checked against rows generated directly from the position-keyed
synthetic scene."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from kinectdepthmapenhancement_b200 import shard, synth


def test_frame_shard_covers_stream():
    for n, world in [(4096, 1), (4096, 8), (10, 4), (3, 8), (0, 2)]:
        spans = [shard.frame_shard(n, world, r) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [b - a for a, b in spans]
        assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard.frame_shard(10, 0, 0)


def test_band_partition_tile_aligned():
    for h, world in [(16384, 8), (16384, 2), (2160, 4), (480, 2), (424, 3), (50, 2)]:
        bands = shard.band_partition(h, world)
        assert bands[0][0] == 0 and bands[-1][1] == h
        assert all(a[1] == b[0] for a, b in zip(bands, bands[1:]))
        assert all(y0 % shard.TILE_H == 0 for y0, _ in bands)
    with pytest.raises(ValueError):
        shard.band_partition(40, 8)
    plan = shard.make_plan(16384, 16384, 9, 3, 8)
    assert plan.up == 11 and plan.down == 11 and plan.band_rows == 2048
    assert plan.halo_bytes_per_direction() == 11 * 16384 * 7      # SURVEY.md 8(e): 1.26 MB
    assert shard.make_plan(640, 480, 7, 0, 2).up == 0 and shard.make_plan(640, 480, 7, 1, 2).down == 0
    with pytest.raises(ValueError):
        shard.make_plan(64, 64, 15, 0, 4)     # 16-row bands thinner than the 17-row halo


def test_synthetic_scene_is_band_decomposable():
    w, h = 96, 80
    d, c = synth.rgbd_frame(w, h, seed=5, frame=2)
    for y0, rows in [(0, 16), (16, 48), (64, 16), (7, 31)]:
        db, cb = synth.rgbd_frame(w, h, seed=5, frame=2, y0=y0, rows=rows)
        assert torch.equal(db, d[y0:y0 + rows]) and torch.equal(cb, c[y0:y0 + rows])


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _halo_worker(rank, world, port, w, h, radius, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        plan = shard.make_plan(w, h, radius, rank, world)
        hx = shard.HaloExchanger(plan, "cpu")
        d, c = synth.rgbd_frame(w, h, seed=11, frame=0, y0=plan.y0, rows=plan.band_rows)
        hx.depth_band.copy_(d)
        hx.bgr_band.copy_(c)
        hx.exchange()
        de, ce = synth.rgbd_frame(w, h, seed=11, frame=0, y0=plan.y0 - plan.up, rows=plan.ext_rows)
        ok = torch.equal(hx.depth_ext, de) and torch.equal(hx.bgr_ext, ce)
        # frame-sharded reduction of per-rank timings: the only collective the stream path uses
        t = torch.tensor([float(rank + 1)], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ok = ok and t.item() == float(world)
        q.put((rank, ok, plan.up, plan.down))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_halo_exchange_gloo(world):
    w, h, radius = 64, 96, 7
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_halo_worker, args=(r, world, port, w, h, radius, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(ok for _, ok, _, _ in res)
    assert res[0][2] == 0 and res[-1][3] == 0 and res[0][3] == radius + 2


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [True, False])
@pytest.mark.parametrize("w,h,radius,world", [(256, 192, 9, 2), (320, 256, 7, 4), (128, 160, 3, 3), (192, 400, 15, 2)])
def test_row_bands_equal_whole_frame_bit_for_bit(w, h, radius, world, overlap):
    """N ranks emulated one after another on one GPU (no waiting kernels): every rank's extended arrays
    are filled as the halo exchange would fill them, the band results are concatenated and must equal
    the single-GPU whole-frame result bit for bit."""
    from kinectdepthmapenhancement_b200 import JointBilateralFilter
    d, c = synth.rgbd_frame(w, h, seed=3, frame=radius)
    # a pixel's arithmetic does not depend on the tile it falls in, so the whole frame (whatever tile
    # height the scheduler picks for it) and the bands (whatever they pick) must agree bit for bit
    full = JointBilateralFilter(w, h, window_radius=radius)
    full.Process(d.cuda(), c.cuda())
    want = full.getFiltered_Device().cpu()
    got = torch.empty_like(want)
    for rank in range(world):
        rb = shard.RowBandJBF(w, h, radius, rank, world)
        p = rb.plan
        rb.halo.depth_ext.copy_(d[p.y0 - p.up:p.y1 + p.down])
        rb.halo.bgr_ext.copy_(c[p.y0 - p.up:p.y1 + p.down])
        got[p.y0:p.y1] = rb.process(exchange=False, overlap=overlap).cpu()   # overlap: interior first, seam strips after
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,radius,world", [(256, 192, 9, 2), (320, 256, 7, 4), (192, 400, 15, 3)])
def test_peer_memory_halos_equal_whole_frame_bit_for_bit(w, h, radius, world):
    """The peer-memory form (halo rows read from the neighbours' bands inside the kernels) emulated on one
    GPU: every rank's arrays hold ONLY its band (halo rows poisoned with NaN / 255 to prove they are never
    read) and the 'peer' pointers point into the other ranks' arrays on the same device."""
    from kinectdepthmapenhancement_b200 import JointBilateralFilter
    d, c = synth.rgbd_frame(w, h, seed=4, frame=radius)
    full = JointBilateralFilter(w, h, window_radius=radius)
    full.Process(d.cuda(), c.cuda())
    want = full.getFiltered_Device().cpu()
    ranks = [shard.RowBandJBF(w, h, radius, r, world) for r in range(world)]
    for rb in ranks:
        p = rb.plan
        rb.halo.depth_ext.fill_(float("nan"))
        rb.halo.bgr_ext.fill_(255)
        rb.depth_band.copy_(d[p.y0:p.y1])
        rb.bgr_band.copy_(c[p.y0:p.y1])
    got = torch.empty_like(want)
    for r, rb in enumerate(ranks):
        p = rb.plan
        d_up = d_dn = b_up = b_dn = 0
        if r > 0:
            q = ranks[r - 1]
            first = q.plan.up + q.plan.band_rows - p.up
            d_up = q.halo.depth_ext.data_ptr() + first * w * 4
            b_up = q.halo.bgr_ext.data_ptr() + first * w * 3
        if r < world - 1:
            q = ranks[r + 1]
            d_dn = q.halo.depth_ext.data_ptr() + q.plan.up * w * 4
            b_dn = q.halo.bgr_ext.data_ptr() + q.plan.up * w * 3
        got[p.y0:p.y1] = rb.process_peer(barrier=False, pointers=(d_up, d_dn, b_up, b_dn)).cpu()
    assert not torch.isnan(got).any()
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))


def _two_rank_worker(rank, world, port, size, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    from tools import workloads
    out = {}
    for mode in ("nccl", "peer"):
        out[mode] = workloads.bands(size, 9, peer=(mode == "peer"), steps=1, oracle_cols=256)
    if rank == 0:
        q.put(out)
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs on one NVLink box")
def test_real_two_rank_bands_nccl_and_peer_memory():
    """The real thing on two GPUs: NCCL send/recv halos and in-kernel peer-memory halos.  Every rank re-filters
    the rows on both sides of the seam without band logic (bit for bit), rank 0 checks the two seam rows against
    the fp64 CPU oracle."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, 29517, 2048, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for mode in ("nccl", "peer"):
        r = res[mode]
        assert r["seam_rows_bitwise_equal_single_gpu_path"] is True, mode
        assert r["oracle_seam_check"]["mask_mismatches"] == 0 and r["oracle_seam_check"]["max_abs_regular_mm"] <= 1e-3
    assert res["nccl"]["band_digests"] == res["peer"]["band_digests"]
