"""GPU parity: DDGI (K18-K21) and reflections (K12, K14-K17) through the C ABI vs the CPU oracle.

Binary decisions inside the shading (which triangle a ray hits, whether a shadow ray is blocked) are computed with the
deterministic fp32 chain, so hit distances and ray directions are compared exactly; colours are compared with
RMSE <= 1e-3 (BASELINE.json) plus a stated max-abs bound (fp16 storage, libm vs CUDA pow/exp).
"""
import ctypes as C

import numpy as np
import pytest

import oracle as O
import pyhr

pytestmark = pytest.mark.gpu

W, H = 192, 112
SKY = (0.3, 0.4, 0.6)


def f16(a):
    return np.ascontiguousarray(a).view(np.float16).astype(np.float32)


def rmse(a, b):
    return float(np.sqrt(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)))


def close(a, b, name, r=1e-3, m=6e-3):
    """rmse and max-abs bounds, both relative to max(1, |reference|): fp16 images holding values >> 1 (squared probe
    distances up to (1.5 * probe_distance)^2) have an ulp of 2^-10 * value."""
    assert a.shape == b.shape, name
    scale = np.maximum(1.0, np.abs(b))
    d = np.abs(a - b) / scale
    e = float(np.sqrt(np.mean(d.astype(np.float64) ** 2)))
    assert e <= r, f"{name}: rmse {e}"
    assert d.max() <= m, f"{name}: max abs {d.max()}"


def run(scene_kind, n_frames, refl_scale, with_ddgi, light=None, cam=None, pan_from=None, tris=0, W=W, H=H, params=None, record=None):
    """params: hr_reflections_params fields to override (the oracle reads the same structure); record: a list that receives
    the device a-trous and final images of every frame"""
    sc = pyhr.SynthScene(scene_kind, tris)
    ss = O.ShadingScene(sc, brute=sc.n_tris <= 4096)
    bn = pyhr.blue_noise()
    ctx = pyhr.Context(0)
    ctx.set_bluenoise(*bn)
    ctx.build_scene(sc)
    ctx.gbuffer_create(W, H)
    mn, mx = sc.bounds()
    info_ok = True
    dd = pyhr.DDGIPass(ctx, W, H, 0) if with_ddgi else None
    rf = pyhr.ReflectionsPass(ctx, W, H, refl_scale)
    for P in ([dd.params] if dd else []) + [rf.params]:
        P.sky_color[0], P.sky_color[1], P.sky_color[2] = SKY
    for k, v in (params or {}).items():
        setattr(rf.params, k, v)
    odd = None
    if dd:
        dd.params.probe_distance = 4.0 if scene_kind == pyhr.SCENE_SHADOWS_TEST else 12.0
        dd.params.normal_bias = 1.0
        odd = O.DDGIOracle(W, H, 0, dd.params, mn, mx)
    orf = O.ReflectionsOracle(W, H, refl_scale, rf.params)
    f, prev_g = None, O.zero_gbuf_mips(W, H)
    zero = pyhr.GBufferHost(W, H)
    ctx.gbuffer_upload(0, zero)
    ctx.gbuffer_upload(1, zero)
    for i in range(n_frames):
        dx = 0.0 if pan_from is None or i < pan_from else 0.05 * (i - pan_from + 1)
        pos, tgt = cam if cam else ((dx, 14.0, 34.0), (dx, 3.0, 0.0))
        f = pyhr.make_frame(pos, tgt, W, H, prev=f, num_frames=i, light=light)
        g = pyhr.write_gbuffer(sc, f, W, H)
        ctx.gbuffer_upload(f.ping_pong, g)
        cur_g = O.GBufMips(g)
        if dd:
            rot = pyhr.rotation_matrix(0.7 + 1.3 * i, (0.3, 1.0, -0.5))
            dd.render(f, rot)
            odd.render(ss, cur_g, f, rot)
            if i == 0:
                u = dd.uniforms()
                assert bytes(u) == bytes(odd.u), "DDGIUniforms differ"
            dird_c, dird_o = dd.download(1).view(np.uint16), odd.dirdepth
            assert np.array_equal(dird_c, dird_o.reshape(dird_c.shape)), f"frame {i}: probe ray direction / hit distance not exact"
            close(f16(dd.download(0)), O.h2f(odd.radiance).reshape(-1, odd.u.rays_per_probe, 4), f"frame {i} ddgi radiance", 2e-3, 0.05)
            close(f16(dd.download(2)), O.h2f(odd.cur_irr), f"frame {i} irradiance atlas")
            close(f16(dd.download(3)), O.h2f(odd.cur_dep), f"frame {i} depth atlas", 2e-3, 0.05)
            close(f16(dd.download(4)), O.h2f(odd.sample), f"frame {i} ddgi sample")
        rf.render(f, dd)
        orf.render(ss, cur_g, prev_g, f, bn, odd)
        prev_g = cur_g
        rt_c, rt_o = f16(rf.download(0)), O.h2f(orf.rt)
        assert np.array_equal(rt_c[..., 3], rt_o[..., 3]), f"frame {i}: reflection ray length (hit / miss / t) not exact"
        close(rt_c[..., :3], rt_o[..., :3], f"frame {i} reflections ray trace", 1e-3, 0.02)
        assert np.array_equal(rf.download(6), orf.tile_flags), f"frame {i}: reflections tile classification"
        close(f16(rf.download(1)), O.h2f(orf.cur_temporal), f"frame {i} reflections temporal")
        mo_c, mo_o = f16(rf.download(4)), O.h2f(orf.cur_moments)
        assert np.array_equal(mo_c[..., 2], mo_o[..., 2]), f"frame {i}: reflections history length"
        close(mo_c, mo_o, f"frame {i} reflections moments")
        close(f16(rf.download(2)), O.h2f(orf.atrous_out), f"frame {i} reflections a-trous")
        close(f16(rf.download(100)), O.h2f(orf.final), f"frame {i} reflections final")
        if record is not None:
            record.append((rf.download(2), rf.download(100)))
    stats = (float(rt_o[..., :3].mean()), float((rt_o[..., 3] > 0).mean()))
    rf.destroy()
    if dd:
        dd.destroy()
    ctx.close()
    return stats


def test_ddgi_and_reflections_static_then_pan():
    """DDGI (867 probes x 256 rays) + half-res reflections reading the DDGI atlas (sample_gi, rough -> DDGI), 3 static + 2 pan frames."""
    mean, hit_frac = run(pyhr.SCENE_SHADOWS_TEST, 5, 1, True, pan_from=3)
    assert mean > 0.01 and 0.05 < hit_frac < 1.0


def test_reflections_full_res_without_ddgi():
    """reflections alone (ddgi = NULL => sample_gi / approximate_with_ddgi off), full-res (no upsample), point light."""
    light = pyhr.default_light(type=1, position=(2.0, 12.0, 6.0), radius=2.5, intensity=500.0)
    mean, hit_frac = run(pyhr.SCENE_SHADOWS_TEST, 3, 0, False, light=light)
    assert mean > 0.001


def test_reflections_arcade_all_lobes():
    """arcade scene: materials with roughness 0.02 (mirror), 0.2 / 0.5 (GGX) and 0.9 (DDGI lobe) are all present."""
    mean, hit_frac = run(pyhr.SCENE_ARCADE, 3, 1, True, light=pyhr.default_light(rot_x_deg=25.0), cam=((0.0, 9.0, -4.0), (2.0, 7.0, 60.0)), tris=20000)
    assert hit_frac > 0.2


def test_reflections_atrous_variants_agree():
    """K16 implementations (hr_debug_set key 6): 4 / 3 = TMA-staged persistent kernel for steps 1-4 / step 1 (default), 2 = packed fp32x2 + row-interleaved wide
    steps, 1 = packed dense tiles, 0 = scalar kernel.  Same staged values and the same arithmetic in 1-3 => bit-identical; the scalar
    kernel differs by rounding only.  5 iterations (steps 1..16), odd tile counts, all lobes."""
    Wt, Ht = 712, 392
    sc = pyhr.SynthScene(pyhr.SCENE_ARCADE, 20000)
    light = pyhr.default_light(rot_x_deg=25.0)
    outs = {}
    for impl in (4, 3, 2, 1, 0):
        ctx = pyhr.Context(0)
        ctx.lib.hr_debug_set(6, impl)
        ctx.set_bluenoise(*pyhr.blue_noise())
        ctx.build_scene(sc)
        ctx.gbuffer_create(Wt, Ht)
        rf = pyhr.ReflectionsPass(ctx, Wt, Ht, 0)
        rf.params.filter_iterations = 5
        rf.params.sky_color[0], rf.params.sky_color[1], rf.params.sky_color[2] = SKY
        f = None
        for i in range(3):
            f = pyhr.make_frame((0.05 * i, 9.0, -4.0), (2.0, 7.0, 60.0), Wt, Ht, prev=f, num_frames=i, light=light)
            ctx.gbuffer_render(f.ping_pong, f)
            rf.render(f, None)
        outs[impl] = (rf.download(2).copy(), rf.download(100).copy())
        rf.destroy()
        ctx.lib.hr_debug_set(6, 3)
        ctx.close()
    for impl in (4, 2, 1):
        assert np.array_equal(outs[3][0], outs[impl][0]) and np.array_equal(outs[3][1], outs[impl][1]), f"impl 3 vs {impl}"
    close(f16(outs[3][1]), f16(outs[0][1]), "packed vs scalar a-trous", 2e-4, 4e-3)
