"""Row-band sharding (SURVEY.md §8e): N-rank results must be BIT-IDENTICAL to the single-GPU result.

* test_sharded_emulation_*: N ranks emulated on one GPU (one hr_ctx per rank, hr_shard_config), the band exchange done by
  the test through hr_pass_download / hr_pass_upload.  Runs on the single-GPU box.
* test_peer_history_emulation_*: the same N emulated ranks, but linked with hr_shard_link_local: nothing is moved by the
  test — every rank's reprojection kernel pulls history texels from the rank that owns their row (the production
  multi-GPU data path, minus CUDA IPC).  Runs on the single-GPU box.
* test_nccl_*: real one-process-per-GPU run (hr_shard_init): peer history over CUDA IPC / NVLink + the NCCL gather of the
  final output; needs >= 2 GPUs (`gpurun --gpus 2 -- python -m pytest tests/test_gpu_multi.py -m gpu`).
"""
import os
import sys

import numpy as np
import pytest
import torch

import oracle as O  # noqa: F401  (path setup)
import pyhr

pytestmark = pytest.mark.gpu

W, H = 256, 144
SH = dict(temporal=1, atrous=2, moments=4, prev=5, final=100)
AO = dict(temporal=1, blur=2, length=4, final=100)


def frames(n, pan_from=3, vertical=0.0, W=W, H=H):
    f = None
    for i in range(n):
        dx = 0.0 if i < pan_from else 0.05 * (i - pan_from + 1)
        dy = 0.0 if i < pan_from else vertical * (i - pan_from + 1)  # vertical motion: reprojection taps cross band borders
        f = pyhr.make_frame((dx, 14.0 + dy, 34.0), (dx, 3.0 - dy, 0.0), W, H, prev=f, num_frames=i)
        yield f


def make_rank(device, sc, sh_scale, ao_scale, rank=0, world=1, W=W, H=H):
    c = pyhr.Context(device)
    c.set_bluenoise(*pyhr.blue_noise())
    c.build_scene(sc)
    c.gbuffer_create(W, H)
    if world > 1:
        c.shard_config(rank, world)
    return c, pyhr.Pass(c, "shadows", W, H, sh_scale), pyhr.Pass(c, "ao", W, H, ao_scale)


def merge_bands(images, pass_h, world, shift=0):
    """assemble the complete image from each rank's copy: rank r contributes its band (what the NCCL exchange does)"""
    out = images[0].copy()
    for r in range(world):
        b, e = pyhr.shard_rows(pass_h, r, world)
        e2 = out.shape[0] if e >= pass_h else e << shift
        out[b << shift:e2] = images[r][b << shift:e2]
    return out


@pytest.mark.parametrize("world,sh_scale,ao_scale", [(2, 0, 1), (3, 0, 1), (4, 1, 0)])
def test_sharded_emulation_bit_identical(world, sh_scale, ao_scale):
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    ref = make_rank(0, sc, sh_scale, ao_scale)
    ranks = [make_rank(0, sc, sh_scale, ao_scale, r, world) for r in range(world)]
    sh_h, ao_h = H >> sh_scale, H >> ao_scale
    for f in frames(7):
        g = pyhr.write_gbuffer(sc, f, W, H)
        for c, sh, ao in [ref] + ranks:
            c.gbuffer_upload(f.ping_pong, g)
            sh.render(f)
            ao.render(f)
        # exchange: final output + history surfaces
        for name, which, shift in (("prev", SH["prev"], 0), ("moments", SH["moments"], 0), ("final", SH["final"], sh_scale)):
            merged = merge_bands([r[1].download(which) for r in ranks], sh_h, world, shift if name == "final" else 0)
            assert np.array_equal(merged, ref[1].download(which)), f"shadows {name} differs (world={world}, frame {f.num_frames})"
            for r in ranks:
                r[1].upload(which, merged)
        for name, which, shift in (("temporal", AO["temporal"], 0), ("length", AO["length"], 0), ("final", AO["final"], ao_scale)):
            merged = merge_bands([r[2].download(which) for r in ranks], ao_h, world, shift if name == "final" else 0)
            assert np.array_equal(merged, ref[2].download(which)), f"ao {name} differs (world={world}, frame {f.num_frames})"
            for r in ranks:
                r[2].upload(which, merged)
    for c, sh, ao in [ref] + ranks:
        sh.destroy()
        ao.destroy()
        c.close()


# 203x117 (world 3): odd pass widths, a last band that ends in a partial tile, and an odd full-res height for the upsample rows
# of the last band (b1 >= H ? H0)
@pytest.mark.parametrize("world,sh_scale,ao_scale,W,H", [pytest.param(2, 0, 1, W, H, id="2-0-1"), pytest.param(5, 0, 0, W, H, id="5-0-0"),
                                                         pytest.param(8, 1, 1, W, H, id="8-1-1"), pytest.param(3, 1, 1, 203, 117, id="3-1-1-203x117")])
def test_peer_history_emulation_bit_identical(world, sh_scale, ao_scale, W, H):
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    ref = make_rank(0, sc, sh_scale, ao_scale, W=W, H=H)
    ranks = [make_rank(0, sc, sh_scale, ao_scale, r, world, W, H) for r in range(world)]
    for r in range(world):
        for q in range(world):
            if q != r:
                ranks[r][1].link_local(q, ranks[q][1])
                ranks[r][2].link_local(q, ranks[q][2])
    sh_h, ao_h = H >> sh_scale, H >> ao_scale
    # Linked ranks wait for each other inside a frame (the ray masks are traced cooperatively: every rank traces its
    # cost-balanced share of the whole image and pushes it to all peers), so the emulated ranks must be able to run
    # concurrently: one CUDA stream per rank (conftest.py raises CUDA_DEVICE_MAX_CONNECTIONS so they get separate queues).
    streams = [torch.cuda.Stream() for _ in range(world)]
    for f in frames(8, pan_from=2, vertical=0.35, W=W, H=H):
        g = pyhr.write_gbuffer(sc, f, W, H)
        ref[0].gbuffer_upload(f.ping_pong, g)
        ref[1].render(f)
        ref[2].render(f)
        for (c, sh, ao), st in zip(ranks, streams):
            c.gbuffer_upload(f.ping_pong, g, st.cuda_stream)
        for (c, sh, ao), st in zip(ranks, streams):
            sh.render(f, st.cuda_stream)
        for (c, sh, ao), st in zip(ranks, streams):
            ao.render(f, st.cuda_stream)
        torch.cuda.synchronize()
        for r in ranks:  # the complete ray mask is on every rank
            assert np.array_equal(r[1].download(0), ref[1].download(0)), f"shadows mask differs (world={world}, frame {f.num_frames})"
            assert np.array_equal(r[2].download(0), ref[2].download(0)), f"ao mask differs (world={world}, frame {f.num_frames})"
        for name, which, shift in (("prev", SH["prev"], 0), ("moments", SH["moments"], 0), ("final", SH["final"], sh_scale)):
            merged = merge_bands([r[1].download(which) for r in ranks], sh_h, world, shift if name == "final" else 0)
            assert np.array_equal(merged, ref[1].download(which)), f"shadows {name} differs (world={world}, frame {f.num_frames})"
        for name, which, shift in (("temporal", AO["temporal"], 0), ("length", AO["length"], 0), ("final", AO["final"], ao_scale)):
            merged = merge_bands([r[2].download(which) for r in ranks], ao_h, world, shift if name == "final" else 0)
            assert np.array_equal(merged, ref[2].download(which)), f"ao {name} differs (world={world}, frame {f.num_frames})"
    for c, sh, ao in [ref] + ranks:
        sh.destroy()
        ao.destroy()
    for c, sh, ao in [ref] + ranks:
        c.close()


def _nccl_worker(rank, world, uid, result_dir):
    import torch
    torch.cuda.set_device(rank)
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    c = pyhr.Context(rank)
    c.set_bluenoise(*pyhr.blue_noise())
    c.build_scene(sc)
    c.gbuffer_create(W, H)
    c.shard_init(rank, world, uid)
    sh, ao = pyhr.Pass(c, "shadows", W, H, 0), pyhr.Pass(c, "ao", W, H, 1)
    outs = []
    for f in frames(6, vertical=0.35):
        g = pyhr.write_gbuffer(sc, f, W, H)
        c.gbuffer_upload(f.ping_pong, g)
        sh.render(f)
        ao.render(f)
        outs.append((sh.download(100), sh.download(SH["prev"]), sh.download(SH["moments"]), ao.download(100), ao.download(AO["temporal"])))
    np.savez(os.path.join(result_dir, f"rank{rank}.npz"), **{f"f{i}_{j}": a for i, o in enumerate(outs) for j, a in enumerate(o)})
    sh.destroy()
    ao.destroy()
    c.shard_shutdown()
    c.close()


def test_nccl_sharded_matches_single(tmp_path):
    import torch
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    uid = pyhr.shard_unique_id()
    mp.spawn(_nccl_worker, args=(world, uid, str(tmp_path)), nprocs=world, join=True)
    # single-GPU reference in this process
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    c, sh, ao = make_rank(0, sc, 0, 1)
    ref = []
    for f in frames(6, vertical=0.35):
        g = pyhr.write_gbuffer(sc, f, W, H)
        c.gbuffer_upload(f.ping_pong, g)
        sh.render(f)
        ao.render(f)
        ref.append((sh.download(100), sh.download(SH["prev"]), sh.download(SH["moments"]), ao.download(100), ao.download(AO["temporal"])))
    # image j: 0 shadows final (gathered: complete on every rank), 1 prev_image, 2 moments, 3 AO final (gathered, full-res),
    # 4 AO temporal — the history images stay distributed (peer history): each rank holds its own band
    band_h = {1: H, 2: H, 4: H >> 1}
    for r in range(world):
        d = np.load(os.path.join(str(tmp_path), f"rank{r}.npz"))
        for i, o in enumerate(ref):
            for j, a in enumerate(o):
                got = d[f"f{i}_{j}"]
                if j in band_h:
                    b, e = pyhr.shard_rows(band_h[j], r, world)
                    assert np.array_equal(got[b:e], a[b:e]), f"rank {r} frame {i} image {j}: own band differs from the single-GPU result"
                else:
                    assert np.array_equal(got, a), f"rank {r} frame {i} image {j} differs from the single-GPU result"
    sh.destroy()
    ao.destroy()
    c.close()


# ---- reflections: peer history + interleaved cooperative ray trace -----------------------------------------------------------------
RF = dict(rt=0, temporal=1, atrous=2, moments=4, final=100)


def _refl_rank(device, sc, scale, rank=0, world=1, W=W, H=H):
    c = pyhr.Context(device)
    c.set_bluenoise(*pyhr.blue_noise())
    c.build_scene(sc)
    c.gbuffer_create(W, H)
    if world > 1:
        c.shard_config(rank, world)
    p = pyhr.ReflectionsPass(c, W, H, scale)
    p.params.sky_color[0], p.params.sky_color[1], p.params.sky_color[2] = 0.3, 0.4, 0.6
    return c, p


@pytest.mark.parametrize("world,scale,W,H", [pytest.param(2, 0, W, H, id="2-0"), pytest.param(5, 1, W, H, id="5-1"), pytest.param(8, 0, W, H, id="8-0"),
                                             pytest.param(3, 1, 203, 117, id="3-1-203x117")])
def test_peer_history_emulation_reflections(world, scale, W, H):
    """N linked ranks on one GPU (the production multi-GPU data path minus CUDA IPC): every rank traces the 8-row chunks
    c % world == rank of the whole image and pushes them to the ranks that filter those rows; reprojection pulls history
    texels from the owner of their row.  Each rank's band of every stage must be BIT-IDENTICAL to the single-GPU images."""
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    ref = _refl_rank(0, sc, scale, W=W, H=H)
    ranks = [_refl_rank(0, sc, scale, r, world, W, H) for r in range(world)]
    for r in range(world):
        for q in range(world):
            if q != r:
                ranks[r][1].link_local(q, ranks[q][1])
    streams = [torch.cuda.Stream() for _ in range(world)]
    ph = H >> scale
    for f in frames(7, pan_from=2, vertical=0.35, W=W, H=H):
        g = pyhr.write_gbuffer(sc, f, W, H)
        ref[0].gbuffer_upload(f.ping_pong, g)
        ref[1].render(f, None)
        for (c, p), st in zip(ranks, streams):
            c.gbuffer_upload(f.ping_pong, g, st.cuda_stream)
        for (c, p), st in zip(ranks, streams):
            p.render(f, None, st.cuda_stream)
        torch.cuda.synchronize()
        for name, which, shift in (("ray trace", RF["rt"], 0), ("temporal", RF["temporal"], 0), ("moments", RF["moments"], 0), ("a-trous", RF["atrous"], 0),
                                   ("final", RF["final"], scale)):
            merged = merge_bands([r[1].download(which) for r in ranks], ph, world, shift if name == "final" else 0)
            assert np.array_equal(merged, ref[1].download(which)), f"reflections {name} differs (world={world}, frame {f.num_frames})"
    for c, p in [ref] + ranks:
        p.destroy()
    for c, p in [ref] + ranks:
        c.close()


def _nccl_refl_worker(rank, world, uid, result_dir):
    import torch
    torch.cuda.set_device(rank)
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    c = pyhr.Context(rank)
    c.set_bluenoise(*pyhr.blue_noise())
    c.build_scene(sc)
    c.gbuffer_create(W, H)
    c.shard_init(rank, world, uid)
    p = pyhr.ReflectionsPass(c, W, H, 0)
    p.params.sky_color[0], p.params.sky_color[1], p.params.sky_color[2] = 0.3, 0.4, 0.6
    outs = []
    for f in frames(6, vertical=0.35):
        c.gbuffer_render(f.ping_pong, f)
        p.render(f, None)
        outs.append((p.download(100), p.download(RF["temporal"]), p.download(RF["moments"])))
    np.savez(os.path.join(result_dir, f"refl{rank}.npz"), **{f"f{i}_{j}": a for i, o in enumerate(outs) for j, a in enumerate(o)})
    p.destroy()
    c.shard_shutdown()
    c.close()


def test_nccl_sharded_reflections_match_single(tmp_path):
    """one process per GPU: gathered final output complete and identical on every rank, history bands identical"""
    import torch
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    uid = pyhr.shard_unique_id()
    mp.spawn(_nccl_refl_worker, args=(world, uid, str(tmp_path)), nprocs=world, join=True)
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    c, p = _refl_rank(0, sc, 0)
    ref = []
    for f in frames(6, vertical=0.35):
        c.gbuffer_render(f.ping_pong, f)
        p.render(f, None)
        ref.append((p.download(100), p.download(RF["temporal"]), p.download(RF["moments"])))
    for r in range(world):
        d = np.load(os.path.join(str(tmp_path), f"refl{r}.npz"))
        b, e = pyhr.shard_rows(H, r, world)
        for i, o in enumerate(ref):
            assert np.array_equal(d[f"f{i}_0"], o[0]), f"rank {r} frame {i}: gathered final output differs from the single-GPU result"
            for j in (1, 2):
                assert np.array_equal(d[f"f{i}_{j}"][b:e], o[j][b:e]), f"rank {r} frame {i} image {j}: own band differs"
    p.destroy()
    c.close()


def _nccl_ddgi_worker(rank, world, uid, result_dir):
    import torch
    torch.cuda.set_device(rank)
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    c = pyhr.Context(rank)
    c.set_bluenoise(*pyhr.blue_noise())
    c.build_scene(sc)
    c.gbuffer_create(W, H)
    c.shard_init(rank, world, uid)
    dd, rf = pyhr.DDGIPass(c, W, H, 0), pyhr.ReflectionsPass(c, W, H, 1)
    dd.params.probe_distance, dd.params.normal_bias = 4.0, 1.0
    for P in (dd.params, rf.params):
        P.sky_color[0], P.sky_color[1], P.sky_color[2] = 0.3, 0.4, 0.6
    outs = []
    for i, f in enumerate(frames(5, vertical=0.2)):
        c.gbuffer_render(f.ping_pong, f)
        dd.render(f, pyhr.rotation_matrix(0.7 + 1.3 * i, (0.3, 1.0, -0.5)))
        rf.render(f, dd)
        outs.append((dd.download(2), dd.download(3), dd.download(100), rf.download(100)))
    np.savez(os.path.join(result_dir, f"ddgi{rank}.npz"), **{f"f{i}_{j}": a for i, o in enumerate(outs) for j, a in enumerate(o)})
    dd.destroy()
    rf.destroy()
    c.shard_shutdown()
    c.close()


def test_nccl_sharded_ddgi_and_reflections_match_single(tmp_path):
    """DDGI probe stages split by z-slices + atlas all-gather, per-pixel sampling by bands, half-res reflections reading the atlas:
    atlases, DDGI sample and the reflections output are complete on every rank and equal the single-GPU images bit for bit."""
    import torch
    world = min(torch.cuda.device_count(), 8)
    if world < 2:
        pytest.skip("needs >= 2 GPUs")
    import torch.multiprocessing as mp
    uid = pyhr.shard_unique_id()
    mp.spawn(_nccl_ddgi_worker, args=(world, uid, str(tmp_path)), nprocs=world, join=True)
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    c = pyhr.Context(0)
    c.set_bluenoise(*pyhr.blue_noise())
    c.build_scene(sc)
    c.gbuffer_create(W, H)
    dd, rf = pyhr.DDGIPass(c, W, H, 0), pyhr.ReflectionsPass(c, W, H, 1)
    dd.params.probe_distance, dd.params.normal_bias = 4.0, 1.0
    for P in (dd.params, rf.params):
        P.sky_color[0], P.sky_color[1], P.sky_color[2] = 0.3, 0.4, 0.6
    ref = []
    for i, f in enumerate(frames(5, vertical=0.2)):
        c.gbuffer_render(f.ping_pong, f)
        dd.render(f, pyhr.rotation_matrix(0.7 + 1.3 * i, (0.3, 1.0, -0.5)))
        rf.render(f, dd)
        ref.append((dd.download(2), dd.download(3), dd.download(100), rf.download(100)))
    names = ("irradiance atlas", "depth atlas", "ddgi sample", "reflections final")
    for r in range(world):
        d = np.load(os.path.join(str(tmp_path), f"ddgi{r}.npz"))
        for i, o in enumerate(ref):
            for j, a in enumerate(o):
                assert np.array_equal(d[f"f{i}_{j}"], a), f"rank {r} frame {i}: {names[j]} differs from the single-GPU result"
    dd.destroy()
    rf.destroy()
    c.close()
