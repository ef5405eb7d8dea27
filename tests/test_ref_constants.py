"""The oracle pinned to the only data the reference holds for this path: its in-source tables and constants.

tests/golden/ref_constants.json is produced by tests/golden/make_ref_constants.py, which parses the literals out of
/root/reference (gi_border_update.glsl:35-143, shadows_denoise_atrous.comp:69-72,99-100 + the reflections twin,
random.glsl:17-56, common.glsl:16-28, reprojection.glsl:6-7, scene_descriptor_set.glsl:202, the struct initialisers of
ray_traced_*.h / ddgi.h).  Here:
  * the oracle's generated border-copy tables equal the reference's two literal tables entry by entry;
  * every named constant of oracle/orc_constants.h equals the parsed value (as binary32);
  * known-answer tests computed in numpy FROM THE PARSED VALUES ONLY (no oracle code) pin the RNG and the a-trous kernels;
  * the ABI's default parameter blocks and struct sizes equal the reference's initialisers.
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

import oracle as O
import pyhr

HERE = os.path.dirname(os.path.abspath(__file__))
REF = json.load(open(os.path.join(HERE, "golden", "ref_constants.json")))


def _orc_const(name, n=6):
    L = O.lib()
    L.orc_get_constant.restype = C.c_int
    L.orc_get_constant.argtypes = [C.c_char_p, C.POINTER(C.c_double), C.c_int]
    buf = (C.c_double * n)()
    cnt = L.orc_get_constant(name.encode(), buf, n)
    assert cnt > 0, f"oracle has no constant named {name}"
    return [buf[i] for i in range(cnt)]


@pytest.mark.parametrize("side,key", [(16, "gi_border_offsets_depth_16"), (8, "gi_border_offsets_irradiance_8")])
def test_border_offset_tables_equal_reference(side, key):
    L = O.lib()
    L.orc_border_offsets.restype = C.c_int
    L.orc_border_offsets.argtypes = [C.c_int, C.c_void_p]
    n = L.orc_border_offsets(side, None)
    ref = np.array(REF[key]["rows"], np.int32)
    assert n == ref.shape[0] == 4 * side + 4
    got = np.zeros((n, 4), np.int32)
    L.orc_border_offsets(side, O.p(got))
    assert np.array_equal(got, ref), f"generated g_offsets differ from {REF[key]['src']}"


@pytest.mark.parametrize("name", ["M_PI", "EPSILON", "MIRROR_REFLECTIONS_ROUGHNESS_THRESHOLD", "DDGI_REFLECTIONS_ROUGHNESS_THRESHOLD", "NORMAL_DISTANCE",
                                  "PLANE_DISTANCE", "MIN_ROUGHNESS"])
def test_scalar_constants_equal_reference(name):
    assert np.float32(_orc_const(name)[0]) == np.float32(REF[name]["value"]), REF[name]["src"]


def test_atrous_tables_equal_reference():
    for pas in ("shadows", "reflections"):
        assert np.array_equal(np.float32(_orc_const("atrous_kernel_weights")), np.float32(REF[f"{pas}_atrous_kernel_weights"]["value"]))
        assert np.array_equal(np.float32(_orc_const("atrous_variance_kernel")), np.float32(REF[f"{pas}_atrous_variance_kernel"]["value"]).reshape(-1))
        assert np.float32(_orc_const("atrous_eps_variance")[0]) == np.float32(REF[f"{pas}_atrous_eps_variance"]["value"])


def test_rng_constants_equal_reference():
    for k, v in REF["rng"].items():
        want = v["value"] if isinstance(v["value"], list) else [v["value"]]
        assert [int(x) for x in _orc_const(f"rng.{k}")] == want, v["src"]


# ---- known-answer tests computed from the parsed constants only --------------------------------------------------------------
def _ref_rng_floats(x, y, frame, n):
    """random.glsl:17-56 restated in Python with every constant taken from ref_constants.json"""
    R = REF["rng"]
    M32 = 0xFFFFFFFF
    mul = R["star_multiplier"]["value"]
    a, b, c = R["rotl_a"]["value"], R["shift_b"]["value"], R["rotl_c"]["value"]
    x0, s0, m0, s1, m1, s2 = R["hash"]["value"]
    one, fshift = R["float_bits"]["value"]

    def rotl(v, k):
        return ((v << k) | (v >> (32 - k))) & M32

    def hsh(s):
        s = ((s ^ x0) ^ (s >> s0)) & M32
        s = (s * m0) & M32
        s = s ^ (s >> s1)
        s = (s * m1) & M32
        return s ^ (s >> s2)

    sx, sy = hsh(((x << R["seed_shift"]["value"]) | y) & M32), hsh(frame)

    def nxt():
        nonlocal sx, sy
        res = (sx * mul) & M32
        sy ^= sx
        sx = rotl(sx, a) ^ sy ^ ((sy << b) & M32)
        sy = rotl(sy, c)
        return res

    nxt()  # rng_init discards one draw
    out = []
    for _ in range(n):
        u = one | (nxt() >> fshift)
        out.append(np.array([u], np.uint32).view(np.float32)[0] - np.float32(1.0))
    return np.array(out, np.float32)


@pytest.mark.parametrize("x,y,frame", [(0, 0, 0), (5, 17, 3), (255, 4095, 123456), (65535, 65535, 0xFFFFFFFF)])
def test_rng_known_answers(x, y, frame):
    got = np.zeros(16, np.float32)
    O.lib().orc_rng_sequence(x, y, frame, O.p(got), 16)
    assert np.array_equal(got, _ref_rng_floats(x, y, frame, 16))


def _flat_gbuf(W, H, z=10.0):
    """constant normal +Z (oct (0,0)), constant linear depth, mesh id 1, not sky"""
    g = pyhr.GBufferHost(W, H)
    g.gb2[:] = 0
    g3 = np.zeros((H, W, 4), np.float16)
    g3[..., 0], g3[..., 2], g3[..., 3] = 0.5, 1.0, z
    g.gb3[:] = g3.view(np.uint16)
    g.depth[:] = 0.5
    return g


def test_shadows_atrous_known_answer_from_reference_kernels():
    """A variance impulse next to a visibility edge: every factor of the filter weight is exercised and the expected
    value is computed here from the reference's parsed kernel tables (shadows_denoise_atrous.comp:94-174,
    edge_stopping.glsl:31-62) in float64, then compared with the oracle's fp16 output."""
    W = H = 16
    kw = REF["shadows_atrous_kernel_weights"]["value"]
    vk = REF["shadows_atrous_variance_kernel"]["value"]
    eps = REF["shadows_atrous_eps_variance"]["value"]
    phi_vis, phi_n, sigma_z = REF["defaults"]["shadows"]["phi_visibility"]["value"], REF["defaults"]["shadows"]["phi_normal"]["value"], REF["defaults"]["shadows"]["sigma_depth"]["value"]
    mips = O.GBufMips(_flat_gbuf(W, H), 1)  # keeps the arrays alive while the oracle reads them
    g = mips.c(0)
    img = np.zeros((H, W, 2), np.float16)
    img[..., 0] = 0.25
    img[:, 9:, 0] = 0.75      # visibility edge between columns 8 and 9
    img[7, 9, 1] = 0.5        # variance impulse on the right of the centre pixel (8, 7)
    img[6, 7, 1] = 0.125      # and one diagonal neighbour
    tf = np.ones((2, 2), np.uint8)
    out = np.zeros((H, W, 2), np.uint16)
    src = np.ascontiguousarray(img.view(np.uint16))
    O.lib().orc_shadows_atrous(C.byref(g), O.p(src), O.p(tf), 1, 1, phi_vis, phi_n, sigma_z, 0.0, O.p(out))
    f = img.astype(np.float64)
    cx, cy = 8, 7
    var_c = sum(vk[abs(dx)][abs(dy)] * f[cy + dy, cx + dx, 1] for dy in (-1, 0, 1) for dx in (-1, 0, 1))
    phi_l = phi_vis * np.sqrt(max(0.0, eps + var_c))
    sw, s0, s1 = 1.0, f[cy, cx, 0], f[cy, cx, 1]
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            if dx == 0 and dy == 0:
                continue
            sv, svar = f[cy + dy, cx + dx]
            w_l = abs(f[cy, cx, 0] - sv) / phi_l
            w_z = np.exp(-0.0 / sigma_z)                       # equal depths; fed into the outer exp as in edge_stopping.glsl:47-59
            w = np.exp(0.0 - max(w_l, 0.0) - max(w_z, 0.0)) * 1.0 ** phi_n
            wk = w * kw[abs(dx)] * kw[abs(dy)]
            sw += wk
            s0 += wk * sv
            s1 += wk * wk * svar
    want = np.array([s0 / sw, s1 / (sw * sw)])
    got = O.h2f(out)[cy, cx].astype(np.float64)
    assert np.allclose(got, want, rtol=2e-3, atol=1e-6), (got, want)


def test_reflections_atrous_known_answer_from_reference_kernels():
    W = H = 16
    kw = REF["reflections_atrous_kernel_weights"]["value"]
    vk = REF["reflections_atrous_variance_kernel"]["value"]
    eps = REF["reflections_atrous_eps_variance"]["value"]
    D = REF["defaults"]["reflections"]
    phi_c, phi_n, sigma_z = D["phi_color"]["value"], D["phi_normal"]["value"], D["sigma_depth"]["value"]
    mips = O.GBufMips(_flat_gbuf(W, H), 1)  # keeps the arrays alive while the oracle reads them
    g = mips.c(0)
    img = np.zeros((H, W, 4), np.float16)
    img[..., :3] = (0.2, 0.3, 0.1)
    img[:, 9:, :3] = (0.6, 0.5, 0.4)
    img[7, 9, 3] = 0.5
    img[6, 7, 3] = 0.125
    tf = np.ones((2, 2), np.uint8)
    out = np.zeros((H, W, 4), np.uint16)
    src = np.ascontiguousarray(img.view(np.uint16))
    O.lib().orc_reflections_atrous(C.byref(g), O.p(src), O.p(tf), 1, 1, phi_c, phi_n, sigma_z, 0, O.p(out))
    f = img.astype(np.float64)

    def lum(c):
        return max(c[0] * 0.299 + c[1] * 0.587 + c[2] * 0.114, 0.0001)

    cx, cy = 8, 7
    var_c = sum(vk[abs(dx)][abs(dy)] * f[cy + dy, cx + dx, 3] for dy in (-1, 0, 1) for dx in (-1, 0, 1))
    phi_l = phi_c * np.sqrt(max(0.0, eps + var_c))
    sw, acc = 1.0, f[cy, cx].copy()
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            if dx == 0 and dy == 0:
                continue
            s = f[cy + dy, cx + dx]
            w = np.exp(0.0 - abs(lum(f[cy, cx]) - lum(s)) / phi_l - np.exp(-0.0 / sigma_z))
            wk = w * kw[abs(dx)] * kw[abs(dy)]
            sw += wk
            acc[:3] += wk * s[:3]
            acc[3] += wk * wk * s[3]
    want = np.array([acc[0] / sw, acc[1] / sw, acc[2] / sw, acc[3] / (sw * sw)])
    got = O.h2f(out)[cy, cx].astype(np.float64)
    assert np.allclose(got, want, rtol=2e-3, atol=1e-6), (got, want)


# ---- the ABI mirrors the reference's initialisers ---------------------------------------------------------------------------------
def _check_defaults(struct, ref):
    for k, v in ref.items():
        got = getattr(struct, k)
        want = v["value"]
        if isinstance(want, bool):
            assert bool(got) == want, (k, v["src"])
        elif isinstance(want, int):
            assert int(got) == want, (k, v["src"])
        else:
            assert np.float32(got) == np.float32(want), (k, got, v["src"])


def test_abi_defaults_equal_reference_initialisers():
    lib = pyhr.load_product()
    sp, ap, rp, dp = pyhr.hr_shadows_params(), pyhr.hr_ao_params(), pyhr.hr_reflections_params(), pyhr.hr_ddgi_params()
    lib.hr_shadows_default_params(C.byref(sp))
    lib.hr_ao_default_params(C.byref(ap))
    lib.hr_reflections_default_params(C.byref(rp))
    lib.hr_ddgi_default_params(C.byref(dp))
    D = REF["defaults"]
    _check_defaults(sp, D["shadows"])
    _check_defaults(ap, D["ao"])
    _check_defaults(rp, D["reflections"])
    _check_defaults(dp, D["ddgi"])


def test_ubo_size_equals_reference_member_list():
    u = REF["ubo_layout"]
    assert C.sizeof(pyhr.hr_ubo) == u["bytes"] == 416, u
