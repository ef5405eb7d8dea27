"""GPU parity tests: CUDA path (through the C ABI) vs the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star): visibility masks bit-exact; floating-point outputs <= 1e-3 RMSE; in addition a
max-abs bound per stage is stated here.  Intermediates are stored as fp16 like the reference's RG16F/RGBA16F images,
so one fp16 ulp (<= 4.9e-4 for values in [0.5,1], 9.8e-4 in [1,2]) is the granularity of any difference.
"""
import numpy as np
import pytest

import oracle as O
import pyhr

pytestmark = pytest.mark.gpu


def f16(a):
    return np.ascontiguousarray(a).view(np.float16).astype(np.float32)


def rmse(a, b):
    return float(np.sqrt(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)))


@pytest.fixture(scope="module")
def ctx():
    c = pyhr.Context(0)
    c.set_bluenoise(*pyhr.blue_noise())
    yield c
    c.close()


def camera_path(i, pan_from=None):
    """static camera, then a lateral pan of 0.05 world units / frame (SURVEY.md §8d)"""
    dx = 0.0 if pan_from is None or i < pan_from else 0.05 * (i - pan_from + 1)
    return (dx, 14.0, 34.0), (dx, 3.0, 0.0)


def run_sequence(ctx, scene_kind, W, H, n_frames, sh_scale, ao_scale, pan_from=None, visible_kind=None, cam=None, check=None, light=None, sh_params=None,
                 ao_params=None):
    """sh_params / ao_params: hr_shadows_params / hr_ao_params fields to override, on the device pass and the oracle alike"""
    bn = pyhr.blue_noise()
    sc = pyhr.SynthScene(scene_kind)
    vis_sc = sc if visible_kind is None else pyhr.SynthScene(visible_kind)
    tri, _ = sc.world_triangles()
    osc = O.Scene(tri, brute=sc.n_tris <= 4096)
    import ctypes as C
    scene_h = ctx.build_scene(sc)
    # fresh g-buffer per sequence: recreate the context-level buffers by using a new context when the size changes
    sh, ao = pyhr.Pass(ctx, "shadows", W, H, sh_scale), pyhr.Pass(ctx, "ao", W, H, ao_scale)
    osh, oao = O.ShadowsOracle(W, H, sh_scale), O.AOOracle(W, H, ao_scale)
    for over, passes in ((sh_params, (sh, osh)), (ao_params, (ao, oao))):
        for k, v in (over or {}).items():
            for x in passes:
                setattr(x.params, k, v)
    f, prev_g = None, O.zero_gbuf_mips(W, H)
    # the device history slot must start as zeros too
    zero = pyhr.GBufferHost(W, H)
    ctx.gbuffer_upload(0, zero)
    ctx.gbuffer_upload(1, zero)
    stats = []
    for i in range(n_frames):
        pos, tgt = cam(i) if cam else camera_path(i, pan_from)
        f = pyhr.make_frame(pos, tgt, W, H, prev=f, num_frames=i, light=light)
        g = pyhr.write_gbuffer(vis_sc, f, W, H)
        ctx.gbuffer_upload(f.ping_pong, g)
        sh.render(f)
        ao.render(f)
        cur_g = O.GBufMips(g)
        osh.render(osc, cur_g, prev_g, f, bn)
        oao.render(osc, cur_g, prev_g, f, bn)
        prev_g = cur_g
        if check:
            check(i, sh, ao, osh, oao, stats)
    sh.destroy()
    ao.destroy()
    ctx.lib.hr_scene_destroy(scene_h)
    return stats


def check_all(i, sh, ao, osh, oao, stats):
    # ---- shadows ----
    assert np.array_equal(sh.download(pyhr_out("SH_RT")), osh.mask), f"frame {i}: shadow mask not bit-exact"
    assert np.array_equal(sh.download(6), osh.tile_flags), f"frame {i}: shadow tile classification differs"
    t_c, t_o = f16(sh.download(1)), O.h2f(osh.temporal)
    m_c, m_o = f16(sh.download(4)), O.h2f(osh.cur_moments)
    assert np.array_equal(m_c[..., 2], m_o[..., 2]), f"frame {i}: history length differs"
    assert np.abs(t_c - t_o).max() <= 2e-3 and rmse(t_c, t_o) <= 1e-3, f"frame {i}: temporal {np.abs(t_c - t_o).max()}"
    assert np.abs(m_c - m_o)[..., :2].max() <= 2e-3
    a_c, a_o = f16(sh.download(2)), O.h2f(osh.atrous_out)
    p_c, p_o = f16(sh.download(5)), O.h2f(osh.prev_image)
    assert rmse(a_c, a_o) <= 1e-3 and np.abs(a_c - a_o).max() <= 4e-3, f"frame {i}: a-trous rmse {rmse(a_c, a_o)} max {np.abs(a_c - a_o).max()}"
    assert rmse(p_c, p_o) <= 1e-3 and np.abs(p_c - p_o).max() <= 4e-3
    fin_c, fin_o = f16(sh.download(100)), O.h2f(osh.final)
    assert fin_c.shape == fin_o.shape
    assert rmse(fin_c, fin_o) <= 1e-3
    # ---- ao ----
    assert np.array_equal(ao.download(0), oao.mask), f"frame {i}: AO mask not bit-exact"
    assert np.array_equal(ao.download(6), oao.tile_flags), f"frame {i}: AO tile classification differs"
    assert np.array_equal(f16(ao.download(4)), O.h2f(oao.cur_length))
    t_c, t_o = f16(ao.download(1)), O.h2f(oao.temporal)
    assert np.abs(t_c - t_o).max() <= 2e-3 and rmse(t_c, t_o) <= 1e-3
    b_c, b_o = f16(ao.download(2)), O.h2f(oao.blur[1])
    assert rmse(b_c, b_o) <= 1e-3 and np.abs(b_c - b_o).max() <= 4e-3, f"frame {i}: blur {np.abs(b_c - b_o).max()}"
    fin_c, fin_o = f16(ao.download(100)), O.h2f(oao.final)
    assert fin_c.shape == fin_o.shape
    assert rmse(fin_c, fin_o) <= 1e-3 and np.abs(fin_c - fin_o).max() <= 4e-3
    stats.append((rmse(a_c, a_o), rmse(fin_c, fin_o)))


def pyhr_out(name):
    return {"SH_RT": 0}[name]


@pytest.fixture(scope="module")
def ctx_256():
    c = pyhr.Context(0)
    c.set_bluenoise(*pyhr.blue_noise())
    c.gbuffer_create(256, 144)
    yield c
    c.close()


def test_shadows_ao_static_then_pan(ctx_256):
    """8 static frames (history builds up) then 4 panning frames (bilinear reprojection, disocclusion), full-res shadows,
    half-res AO + upsample: every intermediate image of both chains against the oracle."""
    stats = run_sequence(ctx_256, pyhr.SCENE_SHADOWS_TEST, 256, 144, 12, 0, 1, pan_from=8, check=check_all)
    assert len(stats) == 12


def test_half_res_shadows_quarter_res_ao(ctx_256):
    """RayTraceScale HALF / QUARTER: mip addressing, upsample kernels, pass sizes that are not multiples of the tile size
    (64x36: 36 % 8 != 0)."""
    run_sequence(ctx_256, pyhr.SCENE_SHADOWS_TEST, 256, 144, 4, 1, 2, pan_from=2, check=check_all)


def test_config1_single_triangle():
    """BASELINE config 1: 256x256 analytic ground plane, single-triangle BVH, 1 spp shadows, no denoise; mask bit-exact."""
    c = pyhr.Context(0)
    c.set_bluenoise(*pyhr.blue_noise())
    c.gbuffer_create(256, 256)
    bn = pyhr.blue_noise()
    occl, ground = pyhr.SynthScene(pyhr.SCENE_SINGLE_TRIANGLE), pyhr.SynthScene(pyhr.SCENE_GROUND_PLANE)
    tri, _ = occl.world_triangles()
    osc = O.Scene(tri, brute=True)
    c.build_scene(occl)
    sh = pyhr.Pass(c, "shadows", 256, 256, 0)
    sh.params.denoise = 0
    osh = O.ShadowsOracle(256, 256, 0)
    osh.params.denoise = 0
    f = None
    for i in range(3):
        f = pyhr.make_frame((0, 8, 20), (0, 0, 0), 256, 256, prev=f, num_frames=i)
        g = pyhr.write_gbuffer(ground, f, 256, 256)
        c.gbuffer_upload(f.ping_pong, g)
        sh.render(f)
        cur = O.GBufMips(g)
        osh.render(osc, cur, cur, f, bn)
        m = sh.download(100)
        assert np.array_equal(m, osh.mask)
        lit = sum(bin(int(x)).count("1") for x in m.ravel())
        assert 0 < lit < 256 * 256  # there is a shadow, and it does not cover everything
    sh.destroy()
    c.close()


def test_point_and_spot_lights(ctx_256):
    """fetch_light_properties point / spot branches (lighting.glsl:56-105): masks stay bit-exact."""
    for ltype in (1, 2):
        light = pyhr.default_light(type=ltype, position=(2.0, 12.0, 6.0), radius=2.5, intensity=500.0, rot_x_deg=0.0, rot_y_deg=0.0)

        def chk(i, sh, ao, osh, oao, stats):
            m = sh.download(0)
            assert np.array_equal(m, osh.mask)
            stats.append(int(m.any()))
        stats = run_sequence(ctx_256, pyhr.SCENE_SHADOWS_TEST, 256, 144, 2, 0, 1, check=chk, light=light)
        assert any(stats)


def test_trace_random_rays_vs_bruteforce(ctx_256):
    """LBVH traversal vs the oracle's brute-force loop: any-hit flags, closest t / primitive / barycentrics, all exact."""
    import torch
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    tri, _ = sc.world_triangles()
    osc = O.Scene(tri, brute=True)
    h = ctx_256.build_scene(sc)
    rng = np.random.default_rng(5)
    n = 20000
    mn, mx = sc.bounds()
    o = rng.uniform(mn - 1, mx + 5, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    # a quarter of the rays axis-aligned / grazing (zero direction components exercise the slab test's inf/NaN handling)
    d[: n // 8, 1] = 0.0
    d[n // 8: n // 4, 0] = 0.0
    d[n // 8: n // 4, 2] = 0.0
    d[: n // 4] /= np.maximum(np.linalg.norm(d[: n // 4], axis=1, keepdims=True), 1e-20)
    rays = np.zeros((n, 8), np.float32)
    rays[:, 0:3], rays[:, 3], rays[:, 4:7], rays[:, 7] = o, 0.01, d, rng.choice([7.0, 1e4], n)
    ref_any = osc.trace_any(rays)
    ref_t, ref_p, ref_uv = osc.trace_closest(rays)
    dr = torch.from_numpy(rays).cuda()
    out_any = torch.empty(n, dtype=torch.int32, device="cuda")
    out_t = torch.empty(n, dtype=torch.float32, device="cuda")
    out_p = torch.empty(n, dtype=torch.int32, device="cuda")
    out_uv = torch.empty((n, 2), dtype=torch.float32, device="cuda")
    import ctypes as C
    st = torch.cuda.current_stream().cuda_stream
    L = ctx_256.lib
    ctx_256.check(L.hr_trace_any(ctx_256.h, C.c_void_p(dr.data_ptr()), C.c_size_t(n), C.c_void_p(out_any.data_ptr()), C.c_void_p(st)))
    ctx_256.check(L.hr_trace_closest(ctx_256.h, C.c_void_p(dr.data_ptr()), C.c_size_t(n), C.c_void_p(out_t.data_ptr()), C.c_void_p(out_p.data_ptr()),
                                     C.c_void_p(out_uv.data_ptr()), C.c_void_p(st)))
    torch.cuda.synchronize()
    assert 0.05 < ref_any.mean() < 0.95
    assert np.array_equal(out_any.cpu().numpy().astype(np.uint32), ref_any)
    assert np.array_equal(out_p.cpu().numpy().view(np.uint32), ref_p)
    assert np.array_equal(out_t.cpu().numpy(), ref_t)
    assert np.array_equal(out_uv.cpu().numpy(), ref_uv)
    L.hr_scene_destroy(h)


def check_gbuffer_mips(ctx, W0, H0):
    """host G-buffer of the shadows-test scene uploaded at W0 x H0: the device mips 0-2 equal the oracle's bit for bit"""
    sc = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
    f = pyhr.make_frame((0, 14, 34), (0, 3, 0), W0, H0)
    g = pyhr.write_gbuffer(sc, f, W0, H0)
    ctx.gbuffer_upload(0, g)
    om = O.GBufMips(g)
    for mip in range(3):
        W, H, gb2, gb3, d = om.levels[mip]
        assert np.array_equal(ctx.gbuffer_download(0, mip, 2, W0, H0), gb2), f"mip {mip} ({W}x{H}) gb2"
        assert np.array_equal(ctx.gbuffer_download(0, mip, 3, W0, H0), gb3), f"mip {mip} ({W}x{H}) gb3"
        assert np.array_equal(ctx.gbuffer_download(0, mip, 0, W0, H0), d), f"mip {mip} ({W}x{H}) depth"


def test_gbuffer_mips_match_oracle(ctx_256):
    check_gbuffer_mips(ctx_256, 256, 144)


def test_atrous_tiled_equals_naive_and_oracle_1080p():
    """The shared-memory tiled a-trous kernel against the plain global-memory kernel (same arithmetic modulo fast exp)
    and the oracle on a 1080p frame of the arcade scene, all 4 step sizes."""
    W, H = 1920, 1080
    c = pyhr.Context(0)
    bn = pyhr.blue_noise()
    c.set_bluenoise(*bn)
    c.gbuffer_create(W, H)
    sc = pyhr.SynthScene(pyhr.SCENE_ARCADE, 60000)
    c.build_scene(sc)
    tri, _ = sc.world_triangles()
    osc = O.Scene(tri)
    sh = pyhr.Pass(c, "shadows", W, H, 0)
    osh = O.ShadowsOracle(W, H, 0)
    f, prev_g = None, O.zero_gbuf_mips(W, H)
    outs = {}
    for impl in (1, 0, 3, 13, 23):  # 13 / 23 = packed kernel (3) with dense tiles for every step / interleaved rows for steps 4 and 8
        c.lib.hr_debug_set(1, impl % 10)
        c.lib.hr_debug_set(5, {13: 0, 23: 2}.get(impl, 1))
        sh.reset_history()
        f = None
        c.gbuffer_upload(0, pyhr.GBufferHost(W, H))
        c.gbuffer_upload(1, pyhr.GBufferHost(W, H))
        for i in range(3):
            f = pyhr.make_frame((0, 9, -4), (2, 7, 60), W, H, prev=f, num_frames=i, light=pyhr.default_light(rot_x_deg=25.0))
            g = pyhr.write_gbuffer(sc, f, W, H)
            c.gbuffer_upload(f.ping_pong, g)
            sh.render(f)
            if impl == 1:
                cur_g = O.GBufMips(g)
                osh.render(osc, cur_g, prev_g, f, bn)
                prev_g = cur_g
        outs[impl] = f16(sh.download(100))
    c.lib.hr_debug_set(1, 3)  # back to the defaults (process-wide switches)
    c.lib.hr_debug_set(5, 1)
    assert np.array_equal(sh.download(0), osh.mask)
    # row-interleaved tiles (steps 4, 8) only change which CTA filters which row: same arithmetic per pixel, same bits
    assert np.array_equal(outs[3], outs[13]) and np.array_equal(outs[3], outs[23])
    ref = O.h2f(osh.final)
    assert rmse(outs[1], outs[0]) <= 2e-4 and np.abs(outs[1] - outs[0]).max() <= 2e-3
    assert rmse(outs[3], outs[0]) <= 2e-4 and np.abs(outs[3] - outs[0]).max() <= 2e-3  # packed fp32x2 kernel
    assert rmse(outs[3], ref) <= 1e-3
    assert rmse(outs[1], ref) <= 1e-3
    assert 0.02 < ref[..., 0].mean() < 0.98
    sh.destroy()
    c.close()
