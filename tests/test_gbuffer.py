"""G-buffer producer (SURVEY.md §8 f1): device ray-caster hr_gbuffer_render vs its CPU statement oracle/orc_gbuffer.cpp
(every bit of all four images) and vs the CPU synthetic writer host/synth.cpp the rest of the suite feeds the passes with.

Reference: src/g_buffer.cpp:100-263, src/shaders/g_buffer.frag:47-111 (direction_to_octohedral, compute_motion_vector,
compute_curvature, linear z, mesh id), clears g_buffer.cpp:72-96.
"""
import numpy as np
import pytest

import oracle as O
import pyhr

W, H = 256, 144
CAM = ((0.0, 14.0, 34.0), (0.0, 3.0, 0.0))


def _h(a):
    return np.ascontiguousarray(a).view(np.float16).astype(np.float32)


def _frames(n, pan=0.25):
    f, out = None, []
    for i in range(n):
        pos = (CAM[0][0] + pan * i, CAM[0][1], CAM[0][2])
        f = pyhr.make_frame(pos, CAM[1], W, H, prev=f, num_frames=i)
        out.append(f)
    return out


def test_oracle_gbuffer_matches_synth_writer():
    """Two independent CPU producers (different BVHs, different arithmetic order) agree: same visible mesh on all but a few
    silhouette pixels, depth / normals / motion vectors / linear z to fp32 / fp16 rounding."""
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    ss = O.ShadingScene(sc, brute=False)
    for f in _frames(3)[1:]:
        a = O.gbuffer_render(ss, f, W, H)
        b = pyhr.write_gbuffer(sc, f, W, H)
        ida, idb = _h(a.gb3)[..., 2], _h(b.gb3)[..., 2]
        sky_a, sky_b = a.depth == 1.0, b.depth == 1.0
        same = (ida == idb) & (sky_a == sky_b)
        assert same.mean() > 0.998, same.mean()
        m = same & ~sky_a
        assert np.abs(a.depth[m] - b.depth[m]).max() < 2e-6
        assert np.abs(_h(a.gb2)[m] - _h(b.gb2)[m]).max() < 2e-3       # oct normal + motion vector, fp16 storage
        assert np.abs(_h(a.gb3)[m][:, 3] - _h(b.gb3)[m][:, 3]).max() <= 0.0626  # linear z: fp16 ulp at z in [32, 64) is 1/32
        assert np.array_equal(a.gb1[m], b.gb1[m])
        # clears on sky pixels
        assert np.all(a.gb2[sky_a] == 0) and np.all(_h(a.gb3)[sky_a][:, 3] == -1.0) and np.all(a.gb1[sky_a] == 0)
        # curvature: zero on the flat floor (mesh 0), positive somewhere on the cylinders
        curv = _h(a.gb3)[..., 1]
        assert np.all(curv[(ida == 0) & ~sky_a] == 0.0) and curv.max() > 0.0


def test_motion_vectors_are_zero_for_a_static_camera_and_nonzero_under_pan():
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    ss = O.ShadingScene(sc, brute=False)
    f0 = pyhr.make_frame(CAM[0], CAM[1], W, H)
    f1 = pyhr.make_frame(CAM[0], CAM[1], W, H, prev=f0, num_frames=1)
    g = O.gbuffer_render(ss, f1, W, H)
    assert np.abs(_h(g.gb2)[..., 2:]).max() <= 2e-4  # prev_view_proj == view_proj up to rounding of the two projections
    f2 = pyhr.make_frame((CAM[0][0] + 0.5, CAM[0][1], CAM[0][2]), CAM[1], W, H, prev=f1, num_frames=2)
    g2 = O.gbuffer_render(ss, f2, W, H)
    assert np.abs(_h(g2.gb2)[..., 2][g2.depth != 1.0]).mean() > 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("scene_kind,tris,W,H", [pytest.param(pyhr.SCENE_SHADOWS_TEST, 0, W, H, id=f"{pyhr.SCENE_SHADOWS_TEST}-0"),
                                                 pytest.param(pyhr.SCENE_ARCADE, 20000, W, H, id=f"{pyhr.SCENE_ARCADE}-20000"),
                                                 # odd width, H % 4 != 0: partial curvature quads at the right / bottom edge, mips 101x58 and 50x29
                                                 pytest.param(pyhr.SCENE_ARCADE, 20000, 203, 117, id=f"{pyhr.SCENE_ARCADE}-20000-203x117")])
def test_device_gbuffer_is_bit_exact_against_the_oracle(scene_kind, tris, W, H):
    sc = pyhr.SynthScene(scene_kind, tris)
    ss = O.ShadingScene(sc, brute=False)
    ctx = pyhr.Context(0)
    ctx.set_bluenoise(*pyhr.blue_noise())
    ctx.build_scene(sc)
    ctx.gbuffer_create(W, H)
    cam = CAM if scene_kind == pyhr.SCENE_SHADOWS_TEST else ((0.0, 9.0, -4.0), (2.0, 7.0, 60.0))
    f = None
    for i in range(3):
        f = pyhr.make_frame((cam[0][0] + 0.3 * i, cam[0][1], cam[0][2]), cam[1], W, H, prev=f, num_frames=i)
        ctx.gbuffer_render(f.ping_pong, f)
        ref = O.gbuffer_render(ss, f, W, H)
        mips = O.GBufMips(ref)
        for mip in range(3):
            w, h, r2, r3, rd = mips.levels[mip]
            assert np.array_equal(ctx.gbuffer_download(f.ping_pong, mip, 0, W, H), rd), f"depth frame {i} mip {mip}"
            assert np.array_equal(ctx.gbuffer_download(f.ping_pong, mip, 2, W, H), r2), f"gb2 frame {i} mip {mip}"
            assert np.array_equal(ctx.gbuffer_download(f.ping_pong, mip, 3, W, H), r3), f"gb3 frame {i} mip {mip}"
        assert np.array_equal(ctx.gbuffer_download(f.ping_pong, 0, 1, W, H), ref.gb1), f"gb1 frame {i}"
    ctx.close()


@pytest.mark.gpu
def test_device_gbuffer_row_ranges_compose():
    """A sharded rank renders only the rows it needs: two row ranges give the same image as one full render."""
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    ctx = pyhr.Context(0)
    ctx.set_bluenoise(*pyhr.blue_noise())
    ctx.build_scene(sc)
    ctx.gbuffer_create(W, H)
    f = _frames(2)[1]
    ctx.gbuffer_render(0, f)
    full = [ctx.gbuffer_download(0, 0, k, W, H) for k in range(4)]
    ctx.gbuffer_render(1, f, 0, 64)
    ctx.gbuffer_render(1, f, 64, H)
    for k in range(4):
        assert np.array_equal(ctx.gbuffer_download(1, 0, k, W, H), full[k])
    ctx.close()


@pytest.mark.gpu
def test_passes_on_the_device_gbuffer_match_the_oracle_on_the_same_gbuffer():
    """End to end without any host G-buffer: hr_gbuffer_render -> shadows + AO; the oracle renders from its own statement
    of the G-buffer.  Masks bit-exact, denoised outputs within 1e-3 RMSE."""
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    ss = O.ShadingScene(sc, brute=False)
    bn = pyhr.blue_noise()
    ctx = pyhr.Context(0)
    ctx.set_bluenoise(*bn)
    ctx.build_scene(sc)
    ctx.gbuffer_create(W, H)
    sh, ao = pyhr.Pass(ctx, "shadows", W, H, 0), pyhr.Pass(ctx, "ao", W, H, 1)
    osh, oao = O.ShadowsOracle(W, H, 0), O.AOOracle(W, H, 1)
    prev_g = O.zero_gbuf_mips(W, H)
    for f in _frames(4, pan=0.1):
        ctx.gbuffer_render(f.ping_pong, f)
        sh.render(f)
        ao.render(f)
        cur_g = O.GBufMips(O.gbuffer_render(ss, f, W, H))
        osh.render(ss.scene, cur_g, prev_g, f, bn)
        oao.render(ss.scene, cur_g, prev_g, f, bn)
        prev_g = cur_g
        assert np.array_equal(sh.download(0), osh.mask) and np.array_equal(ao.download(0), oao.mask)
        a, b = _h(sh.download(100))[..., 0], O.h2f(osh.final)[..., 0]
        assert np.sqrt(np.mean((a - b) ** 2)) < 1e-3
        a, b = _h(ao.download(100)), O.h2f(oao.final)
        assert np.sqrt(np.mean((a - b) ** 2)) < 1e-3
    sh.destroy()
    ao.destroy()
    ctx.close()


@pytest.mark.gpu
def test_pipelined_stage_render_equals_direct_render():
    """hr_gbuffer_stage_render (next frame's ray cast on the side stream) + hr_gbuffer_commit_staged == hr_gbuffer_render"""
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    ctx = pyhr.Context(0)
    ctx.set_bluenoise(*pyhr.blue_noise())
    ctx.build_scene(sc)
    ctx.gbuffer_create(W, H)
    fr = _frames(4)
    ctx.gbuffer_stage_render(fr[0])
    for i, f in enumerate(fr):
        ctx.gbuffer_commit_staged(f.ping_pong)
        if i + 1 < len(fr):
            ctx.gbuffer_stage_render(fr[i + 1])
        got = [ctx.gbuffer_download(f.ping_pong, m, k, W, H) for m in (0, 1) for k in range(4)]
        c2 = pyhr.Context(0)
        c2.set_bluenoise(*pyhr.blue_noise())
        c2.build_scene(sc)
        c2.gbuffer_create(W, H)
        c2.gbuffer_render(f.ping_pong, f)
        ref = [c2.gbuffer_download(f.ping_pong, m, k, W, H) for m in (0, 1) for k in range(4)]
        c2.close()
        for a, b in zip(got, ref):
            assert np.array_equal(a, b), f"frame {i}"
    ctx.close()
