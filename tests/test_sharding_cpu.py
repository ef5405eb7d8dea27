"""CPU, world_size-2 gloo: the row-band sharding plan (band + recompute halo per stage, band exchange of final output and
temporal history after every frame) reproduces the unsharded result exactly.

Each rank runs the CPU oracle but trashes, after every stage, the rows a sharded GPU rank would NOT have computed
(oracle._poison with the halos the CUDA host code derives for the default parameters: ray trace +-24, temporal / a-trous
+-16, AO vertical blur +-8; test_reflections_chunks_and_param_halos_gloo takes them from hr_shard_halo_rows for non-default
iteration counts); the bands are then all-gathered with torch.distributed (gloo) exactly like hr_shard_exchange does with NCCL.
If a halo were too small, garbage would leak into a band and the comparison with the unsharded oracle would fail.

test_cooperative_trace_and_distributed_history_gloo restates the production multi-GPU plan (DESIGN.md §9) the same way: the
ray trace is split into arbitrary, frame-varying shares of mask rows that are exchanged into a complete mask (no halo
re-trace), the denoise stages keep their band +- halo, and each rank keeps the temporal history of its own band only and
fetches the peers' rows before the reprojection.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import oracle as O
import pyhr

W, H = 128, 96


def shard_rows(h, rank, world):
    tiles = (h + 7) // 8
    base, rem = divmod(tiles, world)
    t0 = rank * base + min(rank, rem)
    t1 = t0 + base + (1 if rank < rem else 0)
    return min(t0 * 8, h), min(t1 * 8, h)


def test_partition_matches_library():
    for h in (96, 48, 2160, 540):
        for world in (2, 3, 8):
            for r in range(world):
                assert shard_rows(h, r, world) == pyhr.shard_rows(h, r, world)


def _gather_bands(dist, arr, pass_h, rank, world, shift=0):
    """all-gather with unequal bands = one broadcast per owner (what hr_shard_exchange does inside an NCCL group)"""
    import torch
    out = arr.copy()
    for r in range(world):
        b, e = shard_rows(pass_h, r, world)
        b2, e2 = b << shift, (arr.shape[0] if e >= pass_h else e << shift)
        if e2 <= b2:
            continue
        t = torch.from_numpy(np.ascontiguousarray(arr[b2:e2]).view(np.uint8).copy())
        dist.broadcast(t, src=r)
        out[b2:e2] = t.numpy().view(arr.dtype).reshape(arr[b2:e2].shape)
    return out


def _worker(rank, world, port, q, W=W, H=H, radius=1, iters=4):
    """radius / iters: shadows a-trous parameters; the ranks recompute the halos hr_shard_halo_rows derives from them"""
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
        tri, _ = sc.world_triangles()
        osc = O.Scene(tri, brute=True)
        bn = pyhr.blue_noise()
        ref_sh, ref_ao = O.ShadowsOracle(W, H, 0), O.AOOracle(W, H, 1)
        sh, ao = O.ShadowsOracle(W, H, 0), O.AOOracle(W, H, 1)
        for o in (ref_sh, sh):
            o.params.radius, o.params.filter_iterations = radius, iters
        sh.halos = pyhr.shard_halo_rows("shadows", radius, iters)
        sh.band = shard_rows(sh.H, rank, world)
        ao.band = shard_rows(ao.H, rank, world)
        f, prev = None, O.zero_gbuf_mips(W, H)
        for i in range(5):
            dx = 0.0 if i < 2 else 0.08 * (i - 1)
            f = pyhr.make_frame((dx, 14, 34), (dx, 3, 0), W, H, prev=f, num_frames=i)
            cur = O.GBufMips(pyhr.write_gbuffer(sc, f, W, H))
            ref_sh.render(osc, cur, prev, f, bn)
            ref_ao.render(osc, cur, prev, f, bn)
            sh.render(osc, cur, prev, f, bn)
            ao.render(osc, cur, prev, f, bn)
            prev = cur
            pp = f.ping_pong
            # exchange (shadows: prev_image, moments, final; ao: colour, history length, final)
            sh.prev_image[:] = _gather_bands(dist, sh.prev_image, sh.H, rank, world)
            sh.moments[pp][:] = _gather_bands(dist, sh.moments[pp], sh.H, rank, world)
            final_sh = _gather_bands(dist, sh.final, sh.H, rank, world)
            ao.color[pp][:] = _gather_bands(dist, ao.color[pp], ao.H, rank, world)
            ao.length[pp][:] = _gather_bands(dist, ao.length[pp], ao.H, rank, world)
            final_ao = _gather_bands(dist, ao.final, ao.H, rank, world, shift=1)
            for name, a, b in (("shadows final", final_sh, ref_sh.final), ("prev_image", sh.prev_image, ref_sh.prev_image),
                               ("moments", sh.moments[pp], ref_sh.moments[pp]), ("ao final", final_ao, ref_ao.final),
                               ("ao colour", ao.color[pp], ref_ao.color[pp]), ("ao length", ao.length[pp], ref_ao.length[pp])):
                if not np.array_equal(a, b):
                    q.put(f"rank {rank} frame {i}: {name} differs from the unsharded result")
                    return
        q.put("ok")
    finally:
        dist.destroy_process_group()


def _coop_bounds(mh, world, frame):
    """a frame-dependent, deliberately uneven split of the mask rows (stands in for the cost-balanced partition): every rank
    computes the same table from the same inputs, shares are >= 1 row and unrelated to the denoise bands"""
    rng = np.random.default_rng(1000 + frame)
    cuts = np.sort(rng.choice(np.arange(1, mh), size=world - 1, replace=False))
    return [0] + [int(c) for c in cuts] + [mh]


def _worker_coop(rank, world, port, q):
    """Cooperative ray trace + distributed history (the production multi-GPU plan): each rank traces an arbitrary share of
    the mask rows, the shares are exchanged so every rank holds the complete mask, the denoise stages run on band +- halo,
    and the temporal history of a rank is valid on its own band only — the rows a reprojection needs are fetched from
    their owners before the temporal stage (the GPU kernel pulls them texel by texel; here: one gather)."""
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
        tri, _ = sc.world_triangles()
        osc = O.Scene(tri, brute=True)
        bn = pyhr.blue_noise()
        ref_sh, ref_ao = O.ShadowsOracle(W, H, 0), O.AOOracle(W, H, 1)
        sh, ao = O.ShadowsOracle(W, H, 0), O.AOOracle(W, H, 1)
        sh.band = shard_rows(sh.H, rank, world)
        ao.band = shard_rows(ao.H, rank, world)
        state = {"bounds": None}

        def exchange(mask, a, b):
            out = mask.copy()
            bd = state["bounds"]
            for r in range(world):
                t = torch.from_numpy(np.ascontiguousarray(mask[bd[r]:bd[r + 1]]).view(np.uint8).copy())
                dist.broadcast(t, src=r)
                out[bd[r]:bd[r + 1]] = t.numpy().view(np.uint32).reshape(out[bd[r]:bd[r + 1]].shape)
            return out

        sh.mask_exchange = ao.mask_exchange = exchange
        f, prev = None, O.zero_gbuf_mips(W, H)
        for i in range(5):
            dx = 0.0 if i < 2 else 0.08 * (i - 1)
            dy = 0.0 if i < 2 else 0.3 * (i - 1)  # vertical motion: history taps cross the band borders
            f = pyhr.make_frame((dx, 14 + dy, 34), (dx, 3 - dy, 0), W, H, prev=f, num_frames=i)
            cur = O.GBufMips(pyhr.write_gbuffer(sc, f, W, H))
            ref_sh.render(osc, cur, prev, f, bn)
            ref_ao.render(osc, cur, prev, f, bn)
            pp = f.ping_pong
            # history is distributed: before the reprojection, rows owned by the peers are fetched from them
            if i > 0:
                sh.prev_image[:] = _gather_bands(dist, sh.prev_image, sh.H, rank, world)
                sh.moments[1 - pp][:] = _gather_bands(dist, sh.moments[1 - pp], sh.H, rank, world)
                ao.color[1 - pp][:] = _gather_bands(dist, ao.color[1 - pp], ao.H, rank, world)
                ao.length[1 - pp][:] = _gather_bands(dist, ao.length[1 - pp], ao.H, rank, world)
            for o in (sh, ao):
                state["bounds"] = _coop_bounds(o.mask.shape[0], world, i)
                o.rt_share = (state["bounds"][rank], state["bounds"][rank + 1])
                o.render(osc, cur, prev, f, bn)
            prev = cur
            if not (np.array_equal(sh.mask, ref_sh.mask) and np.array_equal(ao.mask, ref_ao.mask)):
                q.put(f"rank {rank} frame {i}: exchanged ray mask is not the complete mask")
                return
            # own band only: trash everything else in the history this rank keeps
            for o, arrs in ((sh, (sh.prev_image, sh.moments[pp])), (ao, (ao.color[pp], ao.length[pp]))):
                for a in arrs:
                    o._poison(a, 0)
            b0, b1 = sh.band
            a0, a1 = ao.band
            checks = (("shadows final", sh.final[b0:b1], ref_sh.final[b0:b1]), ("prev_image", sh.prev_image[b0:b1], ref_sh.prev_image[b0:b1]),
                      ("moments", sh.moments[pp][b0:b1], ref_sh.moments[pp][b0:b1]), ("ao colour", ao.color[pp][a0:a1], ref_ao.color[pp][a0:a1]),
                      ("ao length", ao.length[pp][a0:a1], ref_ao.length[pp][a0:a1]),
                      ("ao final", ao.final[a0 << 1:(ao.final.shape[0] if a1 >= ao.H else a1 << 1)], ref_ao.final[a0 << 1:(ao.final.shape[0] if a1 >= ao.H else a1 << 1)]))
            for name, a, b in checks:
                if not np.array_equal(a, b):
                    q.put(f"rank {rank} frame {i}: {name} (own band) differs from the unsharded result")
                    return
        q.put("ok")
    finally:
        dist.destroy_process_group()


RW, RH = 96, 160  # reflections plan: 20 tiles of 8 rows


def _worker_refl(rank, world, port, q):
    """Reflections, the production plan (hr_reflections_render, DESIGN.md §9): rank r traces the 8-row chunks c % world == r of the
    whole image and the chunks are exchanged; temporal + a-trous run on band +- the halo hr_shard_halo_rows derives from the
    parameters (here 3 and 5 iterations: 8 and 32 rows — not the default); the history (temporal output + moments) of a rank is
    valid on its own band only and the peers' rows are fetched before the reprojection."""
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
        ss = O.ShadingScene(sc, brute=True)
        bn = pyhr.blue_noise()

        def chunk_exchange(img):
            out = img.copy()
            for c in range((RH + 7) // 8):
                t = torch.from_numpy(np.ascontiguousarray(img[c * 8:c * 8 + 8]).view(np.uint8).copy())
                dist.broadcast(t, src=c % world)
                out[c * 8:c * 8 + 8] = t.numpy().view(np.uint16).reshape(out[c * 8:c * 8 + 8].shape)
            return out

        for iters in (3, 5):
            prm = pyhr.hr_reflections_params()
            pyhr.load_product().hr_reflections_default_params(C.byref(prm))
            prm.filter_iterations = iters
            prm.sky_color[0], prm.sky_color[1], prm.sky_color[2] = 0.3, 0.4, 0.6
            ref, o = O.ReflectionsOracle(RW, RH, 0, prm), O.ReflectionsOracle(RW, RH, 0, prm)
            o.band = shard_rows(RH, rank, world)
            o.halos = pyhr.shard_halo_rows("reflections", prm.radius, iters)
            o.rt_chunks, o.rt_exchange = (rank, world), chunk_exchange
            f, prev = None, O.zero_gbuf_mips(RW, RH)
            for i in range(4):
                dy = 0.0 if i < 2 else 0.4 * (i - 1)  # vertical motion: history taps cross the band borders
                f = pyhr.make_frame((0.0, 14 + dy, 34), (0.0, 3 - dy, 0), RW, RH, prev=f, num_frames=i)
                cur = O.GBufMips(pyhr.write_gbuffer(sc, f, RW, RH))
                pp = f.ping_pong
                ref.render(ss, cur, prev, f, bn)
                if i > 0:  # peer history: rows owned by the other ranks come from them
                    o.temporal[1 - pp][:] = _gather_bands(dist, o.temporal[1 - pp], RH, rank, world)
                    o.moments[1 - pp][:] = _gather_bands(dist, o.moments[1 - pp], RH, rank, world)
                o.render(ss, cur, prev, f, bn)
                prev = cur
                final = _gather_bands(dist, o.final, RH, rank, world)
                b0, b1 = o.band
                checks = (("gathered final", final, ref.final), ("temporal (own band)", o.temporal[pp][b0:b1], ref.temporal[pp][b0:b1]),
                          ("moments (own band)", o.moments[pp][b0:b1], ref.moments[pp][b0:b1]))
                for name, a, b in checks:
                    if not np.array_equal(a, b):
                        q.put(f"rank {rank} iterations {iters} frame {i}: {name} differs from the unsharded result")
                        return
                o._poison(o.temporal[pp], 0)  # a rank keeps the history of its own band only
                o._poison(o.moments[pp], 0)
        q.put("ok")
    finally:
        dist.destroy_process_group()


def _run_world(worker, world, *args):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000 + world + (17 if worker is _worker_coop else 0) + (41 if worker is _worker_refl else 0) + (67 if worker is _worker else 0)
    procs = [ctx.Process(target=worker, args=(r, world, port, q) + args) for r in range(world)]
    for p_ in procs:
        p_.start()
    res = [q.get(timeout=600) for _ in range(world)]
    for p_ in procs:
        p_.join(60)
    return res


@pytest.mark.parametrize("world", [2, 3])
def test_cooperative_trace_and_distributed_history_gloo(world):
    assert _run_world(_worker_coop, world) == ["ok"] * world


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_oracle_gloo(world):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000 + world
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p_ in procs:
        p_.start()
    res = [q.get(timeout=600) for _ in range(world)]
    for p_ in procs:
        p_.join(60)
    assert res == ["ok"] * world, res


@pytest.mark.parametrize("radius,iters", [(2, 6), (2, 2)])
def test_sharded_oracle_ragged_param_halos_gloo(radius, iters):
    """203x117 on 3 ranks: the last band ends in a partial tile (rows 80..117) and the shadows halos come from hr_shard_halo_rows
    for a-trous parameters off the defaults (radius 2 with 6 iterations: 128 rows, the whole image; with 2 iterations: 8 rows)"""
    assert _run_world(_worker, 3, 203, 117, radius, iters) == ["ok"] * 3


@pytest.mark.parametrize("world", [2, 3])
def test_reflections_chunks_and_param_halos_gloo(world):
    assert _run_world(_worker_refl, world) == ["ok"] * world


def test_halo_plan_query():
    """hr_shard_halo_rows (pure, no GPU): the recompute halos follow from the parameters"""
    assert pyhr.shard_halo_rows("shadows", 1, 4) == (16, 24)          # 1 + 2 + 4 + 8 + 1 = 16
    assert pyhr.shard_halo_rows("reflections", 1, 5) == (32, 40)      # 31 + 1
    assert pyhr.shard_halo_rows("shadows", 2, 4) == (32, 40)          # 2 * 15 + 1 = 31 -> 32
    assert pyhr.shard_halo_rows("shadows", 1, 0) == (8, 16)           # the upsample's extra coarse row, rounded to a tile
    assert pyhr.shard_halo_rows("ao", blur_radius=5) == (16, 24)
    assert pyhr.shard_halo_rows("ao", blur_radius=12) == (24, 32)
    for it in range(0, 9):
        for rad in (1, 2):
            d, r = pyhr.shard_halo_rows("shadows", rad, it)
            assert d % 8 == 0 and d >= sum(rad << i for i in range(it)) + 1 and r == d + 8
