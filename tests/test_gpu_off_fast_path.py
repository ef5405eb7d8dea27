"""GPU parity off the fast path: the shadows, AO and reflections chains at ragged image sizes and non-default filter parameters
against the CPU oracle.

The a-trous, blur and upsample stages pick their kernel from the pass size and the filter parameters (svgf_atrous.cu
launch_shadows_atrous, svgf_refl_atrous_v2.cu launch_reflections_atrous_v2, svgf_misc_v2.cu launch_ao_blur /
launch_upsample_scalar / launch_upsample_vec4_v2).  The packed / TMA kernels need an even width, radius 1, phi_normal == 32 and
steps <= 8 (16 for reflections); everything else runs the scalar tiled or naive kernels, k_ao_blur_v1 (blur_radius > 8),
k_upsample_v2 (not an exact 2x) or the v1 upsample (full-res width 1).  Odd widths and heights that are not multiples of 4 / 8
also leave partial 2x2 curvature quads, partial 8x4 mask words and partial 8x8 tiles at the right and bottom edges.

Where a debug switch can force the kernel a case is meant to reach, the case is also run with that switch and the two results
must be the same bits: a case that silently took the fast kernel would fail that comparison (test_fast_kernel_differs_from_the_tiled_one
shows that the comparison can fail).  The bars are those of test_gpu_parity / test_gpu_gi_refl; only the 1366x768 arcade runs use
the zero-variance outlier rule of test_gpu_config_sizes.bounded (DESIGN.md §6).
"""
import contextlib

import numpy as np
import pytest

import oracle as O
import pyhr
from test_gpu_config_sizes import _same_gbuffer, check_all_large
from test_gpu_gi_refl import run as run_reflections
from test_gpu_parity import check_all, check_gbuffer_mips, run_sequence

pytestmark = pytest.mark.gpu

# hr_debug_set keys: 1 = shadows a-trous implementation (0 naive, 1 tiled, 3 packed), 6 = reflections a-trous implementation
# (0 scalar, 3 packed + TMA).  Process-wide: always restored to these defaults.
DEBUG_DEFAULTS = {1: 3, 6: 3}


@contextlib.contextmanager
def forced(key, value):
    lib = pyhr.load_product()
    lib.hr_debug_set(key, value)
    try:
        yield
    finally:
        lib.hr_debug_set(key, DEBUG_DEFAULTS[key])


def context(W, H):
    c = pyhr.Context(0)
    c.set_bluenoise(*pyhr.blue_noise())
    c.gbuffer_create(W, H)
    return c


def pass_size(W, H, scale):
    for _ in range(scale):
        W, H = max(W // 2, 1), max(H // 2, 1)
    return W, H


def shadows_forced_impl(W, sh_params):
    """the hr_debug_set(1, .) value that runs the kernels launch_shadows_atrous must pick for these parameters at pass width W
    (steps > 8 run the naive kernel under both), or None when the packed kernel is expected"""
    if sh_params.get("radius", 1) != 1:
        return 0
    if W % 2 or sh_params.get("phi_normal", 32.0) != 32.0:
        return 1
    return None


def shadows_ao(W, H, sh_scale, ao_scale, n_frames, pan_from, sh_params=None, ao_params=None, check=check_all):
    """run_sequence on a fresh context of this size; returns the device images (shadows a-trous / history / final, AO final)
    of every frame"""
    out = []

    def chk(i, sh, ao, osh, oao, stats):
        if check:
            check(i, sh, ao, osh, oao, [])
        out.append([sh.download(2), sh.download(5), sh.download(100), ao.download(100)])

    c = context(W, H)
    try:
        run_sequence(c, pyhr.SCENE_SHADOWS_TEST, W, H, n_frames, sh_scale, ao_scale, pan_from=pan_from, check=chk, sh_params=sh_params, ao_params=ao_params)
    finally:
        c.close()
    return out


def assert_same_images(a, b, what):
    for i, (fa, fb) in enumerate(zip(a, b)):
        for j, (x, y) in enumerate(zip(fa, fb)):
            assert np.array_equal(x, y), f"{what}: frame {i} image {j} is not bit-identical"


def shadows_case(W, H, sh_scale, ao_scale, n_frames=5, pan_from=3, sh_params=None, ao_params=None):
    """every intermediate against the oracle; then, if the shadows pass is off the packed kernel, the same sequence with that
    kernel forced must give the same bits"""
    got = shadows_ao(W, H, sh_scale, ao_scale, n_frames, pan_from, sh_params, ao_params)
    impl = shadows_forced_impl(pass_size(W, H, sh_scale)[0], sh_params or {})
    if impl is not None:
        with forced(1, impl):
            ref = shadows_ao(W, H, sh_scale, ao_scale, n_frames, pan_from, sh_params, ao_params, check=None)
        assert_same_images(got, ref, f"shadows a-trous vs hr_debug_set(1, {impl})")
    return got


# ---- 1. ragged sizes, default parameters ------------------------------------------------------------------------------------------

def test_gbuffer_mips_203x117():
    """odd sizes at every level: mips 101x58 and 50x29 (NEAREST rule of the down-sampling)"""
    c = context(203, 117)
    try:
        check_gbuffer_mips(c, 203, 117)
    finally:
        c.close()


@pytest.mark.parametrize("sh_scale,ao_scale", [(0, 1), (1, 2), (2, 0)])
def test_shadows_ao_203x117(sh_scale, ao_scale):
    """odd W at full and half res, H % 4 != 0, a quarter-res pass that is not an exact 2x (50x29), partial mask words, tiles and
    temporal CTAs; the upsample runs k_upsample_v2.  Odd shadows widths must equal the forced tiled kernel."""
    shadows_case(203, 117, sh_scale, ao_scale, n_frames=6, pan_from=3)


@pytest.mark.parametrize("W,H", [(40, 12), (7, 5)])
@pytest.mark.parametrize("scale", [0, 1, 2])
def test_shadows_ao_smaller_than_a_tile(W, H, scale):
    """images smaller than one 8x8 tile / one 32x8 CTA (7x5 at quarter res is 1x1); 40x12 keeps W even (packed kernel with
    staging boxes larger than the image)"""
    shadows_case(W, H, scale, scale, n_frames=4, pan_from=2)


def test_shadows_ao_width_1_upsample_v1():
    """1x37 at half res: the only configuration whose upsample footprint does not fit k_upsample_v2 (launch_upsample_scalar_v1)"""
    shadows_case(1, 37, 1, 1, n_frames=4, pan_from=2)


@pytest.mark.parametrize("sh_scale", [0, 1])
def test_shadows_ao_1366x768_device_gbuffer(sh_scale):
    """A 1366x768 window: half-res passes are 683x384 (odd width: tiled shadows a-trous, k_ao_blur_v2 at an odd width); arcade
    scene with 20k triangles from the device G-buffer producer, whose mips 0 and 1 must equal the oracle's bit for bit first.
    Pixel values use test_gpu_config_sizes.bounded: at these sizes a few freshly disoccluded zero-variance pixels amplify one
    fp16 ulp (DESIGN.md §6)."""
    W, H = 1366, 768
    light = pyhr.default_light(rot_x_deg=25.0)
    sc = pyhr.SynthScene(pyhr.SCENE_ARCADE, 20000)
    ss = O.ShadingScene(sc, brute=False)
    bn = pyhr.blue_noise()

    def sequence(check):
        ctx = context(W, H)
        ctx.build_scene(sc)
        sh, ao = pyhr.Pass(ctx, "shadows", W, H, sh_scale), pyhr.Pass(ctx, "ao", W, H, 1)
        osh, oao = O.ShadowsOracle(W, H, sh_scale), O.AOOracle(W, H, 1)
        prev_g, f, out = O.zero_gbuf_mips(W, H), None, []
        for i in range(4):  # 2 static frames, 2 pan frames
            dx = 0.0 if i < 2 else 0.05 * (i - 1)
            f = pyhr.make_frame((dx, 9.0, -4.0), (2.0 + dx, 7.0, 60.0), W, H, prev=f, num_frames=i, light=light)
            ctx.gbuffer_render(f.ping_pong, f)
            sh.render(f)
            ao.render(f)
            if check:
                ref = O.gbuffer_render(ss, f, W, H)
                _same_gbuffer(ctx, f, ref, W, H)
                cur_g = O.GBufMips(ref)
                _, _, gb2, gb3, d = cur_g.levels[1]
                for which, arr in ((0, d), (2, gb2), (3, gb3)):
                    assert np.array_equal(ctx.gbuffer_download(f.ping_pong, 1, which, W, H), arr), f"frame {i}: device G-buffer mip 1 image {which}"
                osh.render(ss.scene, cur_g, prev_g, f, bn)
                oao.render(ss.scene, cur_g, prev_g, f, bn)
                prev_g = cur_g
                check_all_large(i, sh, ao, osh, oao)
            out.append([sh.download(2), sh.download(100), ao.download(100)])
        sh.destroy()
        ao.destroy()
        ctx.close()
        return out

    got = sequence(True)
    if sh_scale == 1:  # 683 wide
        with forced(1, 1):
            assert_same_images(got, sequence(False), "1366x768 half-res shadows vs hr_debug_set(1, 1)")


ARCADE_VIEW = dict(light=pyhr.default_light(rot_x_deg=25.0), cam=((0.0, 9.0, -4.0), (2.0, 7.0, 60.0)))


def reflections_case(forced_scalar, **kw):
    """test_gpu_gi_refl.run at this size / with these parameters; with forced_scalar the same sequence under hr_debug_set(6, 0)
    (scalar k_refl_atrous) must give the same bits"""
    got = []
    run_reflections(record=got, **kw)
    if forced_scalar:
        ref = []
        with forced(6, 0):
            run_reflections(record=ref, **kw)
        assert_same_images(got, ref, "reflections a-trous vs hr_debug_set(6, 0)")


@pytest.mark.parametrize("scale", [0, 1])
def test_ddgi_reflections_203x117(scale):
    """odd widths (203 / 101) through K14-K17 (scalar a-trous) and, at half res, the vec4 upsample that is not an exact 2x"""
    reflections_case(True, scene_kind=pyhr.SCENE_SHADOWS_TEST, n_frames=4, refl_scale=scale, with_ddgi=True, pan_from=2, W=203, H=117)


def test_reflections_40x12():
    """even width smaller than one tile / TMA box: the packed and TMA kernels on an image smaller than what they stage"""
    run_reflections(pyhr.SCENE_SHADOWS_TEST, 3, 0, False, pan_from=1, W=40, H=12)


def test_reflections_1366x768_half_res():
    """683x384 reflections (scalar a-trous) on the 20k-triangle arcade scene, upsampled to 1366x768"""
    reflections_case(True, scene_kind=pyhr.SCENE_ARCADE, n_frames=3, refl_scale=1, with_ddgi=False, tris=20000, W=1366, H=768, **ARCADE_VIEW)


# ---- 2. non-default parameters ----------------------------------------------------------------------------------------------------

SIZES = [(192, 112), (203, 117)]

SHADOW_PARAMS = {
    "radius2": {"radius": 2},
    "radius2_iter6_feedback5": {"radius": 2, "filter_iterations": 6, "feedback_iteration": 5},
    "iter0": {"filter_iterations": 0},
    "iter5": {"filter_iterations": 5},
    "iter8": {"filter_iterations": 8},  # steps up to 128: more than the image
    "feedback0": {"feedback_iteration": 0},
    "feedback_last": {"feedback_iteration": 3},  # = filter_iterations - 1: filtered into atrous[], then copied to the history
    "feedback_none": {"feedback_iteration": 4},  # >= filter_iterations: the history keeps last frame's image
    "phi_normal16": {"phi_normal": 16.0},
    "phi_normal64": {"phi_normal": 64.0},
    "power1": {"power": 1.0},
}


@pytest.mark.parametrize("W,H", SIZES)
@pytest.mark.parametrize("name", list(SHADOW_PARAMS))
def test_shadows_parameters(name, W, H):
    """shadows a-trous off its defaults (full-res shadows, half-res AO); radius 2 must equal the forced naive kernel,
    phi_normal != 32 and odd widths the forced tiled one"""
    shadows_case(W, H, 0, 1, sh_params=SHADOW_PARAMS[name])


@pytest.mark.parametrize("W,H", SIZES)
@pytest.mark.parametrize("blur_radius", [1, 8, 9, 16])
def test_ao_blur_radius(blur_radius, W, H):
    """blur_radius 1..8 runs k_ao_blur_v2, 9..16 k_ao_blur_v1 (8 and 9 sit either side of the switch)"""
    shadows_case(W, H, 0, 1, ao_params={"blur_radius": blur_radius})


REFLECTION_PARAMS = {
    "iter0": ({"filter_iterations": 0}, False),
    "iter5": ({"filter_iterations": 5}, False),
    "phi_normal16": ({"phi_normal": 16.0}, False),
    "blur_as_input_feedback0": ({"blur_as_input": 1, "feedback_iteration": 0}, False),
    "blur_as_input_feedback3": ({"blur_as_input": 1, "feedback_iteration": 3}, False),
    "no_sample_gi": ({"sample_gi": 0}, True),
    "no_approximate_with_ddgi": ({"approximate_with_ddgi": 0}, True),
}


@pytest.mark.parametrize("W,H", SIZES)
@pytest.mark.parametrize("name", list(REFLECTION_PARAMS))
def test_reflections_parameters(name, W, H):
    """half-res reflections off their defaults; odd widths and phi_normal != 32 must equal the forced scalar a-trous kernel"""
    params, ddgi = REFLECTION_PARAMS[name]
    scalar = W // 2 % 2 == 1 or params.get("phi_normal", 32.0) != 32.0
    reflections_case(scalar, scene_kind=pyhr.SCENE_SHADOWS_TEST, n_frames=4, refl_scale=1, with_ddgi=ddgi, pan_from=2, W=W, H=H, params=params)


# ---- 3. the forced-kernel comparisons can fail ------------------------------------------------------------------------------------

def test_fast_kernel_differs_from_the_tiled_one():
    """At an even width with default parameters the packed kernel runs, and its bits differ from the forced tiled kernel's:
    the bit-identity checks above do tell the kernels apart."""
    fast = shadows_ao(192, 112, 0, 1, 3, None, check=None)
    with forced(1, 1):
        tiled = shadows_ao(192, 112, 0, 1, 3, None, check=None)
    assert any(not np.array_equal(a[0], b[0]) for a, b in zip(fast, tiled)), "packed and tiled a-trous gave the same bits"
    got = []
    run_reflections(pyhr.SCENE_SHADOWS_TEST, 3, 1, False, W=192, H=112, record=got)
    ref = []
    with forced(6, 0):
        run_reflections(pyhr.SCENE_SHADOWS_TEST, 3, 1, False, W=192, H=112, record=ref)
    assert any(not np.array_equal(a[0], b[0]) for a, b in zip(got, ref)), "packed and scalar reflections a-trous gave the same bits"
