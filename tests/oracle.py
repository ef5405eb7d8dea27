"""ctypes binding + host sequencing for the CPU oracle (oracle/_build/liboracle.so).  TEST INFRASTRUCTURE ONLY.

`ShadowsOracle` / `AOOracle` replay RayTracedShadows::render (src/ray_traced_shadows.cpp:100-116, :938-1255) and
RayTracedAO::render (src/ray_traced_ao.cpp:98-112, :829-1137) on the oracle's stage functions, with the same
ping-pong / history bookkeeping (SURVEY.md Appendix B).
"""
import ctypes as C
import os
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hybrid-rendering_b200"))
import pyhr  # noqa: E402

LIB_ORACLE = os.path.join(ROOT, "oracle", "_build", "liboracle.so")


class orc_gbuf(C.Structure):
    _fields_ = [("W", C.c_int32), ("H", C.c_int32), ("gb2", C.c_void_p), ("gb3", C.c_void_p), ("depth", C.c_void_p)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_ORACLE):
            raise RuntimeError(f"{LIB_ORACLE} missing: run `make -C {ROOT}/oracle`")
        L = C.CDLL(LIB_ORACLE)
        L.orc_scene_create.restype = C.c_void_p
        L.orc_scene_create.argtypes = [C.c_void_p, C.c_size_t, C.c_int]
        L.orc_scene_destroy.argtypes = [C.c_void_p]
        L.orc_scene_set_brute.argtypes = [C.c_void_p, C.c_int]
        L.orc_trace_any.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.orc_trace_closest.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_det_sincos.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        L.orc_oct_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
        L.orc_sample_blue_noise.restype = C.c_float
        L.orc_sample_blue_noise.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        L.orc_build_mip.argtypes = [C.c_int, C.c_int] + [C.c_void_p] * 6
        P = C.c_void_p
        F = C.c_float
        I = C.c_int
        L.orc_shadows_ray_trace.argtypes = [P, P, P, F, P, P, P]
        L.orc_ao_ray_trace.argtypes = [P, P, P, F, F, P, P, P]
        L.orc_shadows_temporal.argtypes = [P, P, P, P, P, P, F, F, P, P, P]
        L.orc_shadows_atrous.argtypes = [P, P, P, I, I, F, F, F, F, P]
        L.orc_upsample_scalar.argtypes = [P, P, P, I, F, F, P]
        L.orc_ao_temporal.argtypes = [P, P, P, P, P, P, F, P, P, P]
        L.orc_ao_bilateral_blur.argtypes = [P, P, P, P, I, I, I, P]
        L.orc_shadows_ray_trace_spp.argtypes = [P, P, P, F, I, P, P, P]
        L.orc_ao_ray_trace_spp.argtypes = [P, P, P, F, F, I, P, P, P]
        L.orc_shadows_temporal_spp.argtypes = [P, P, P, I, P, P, P, F, F, P, P, P]
        L.orc_ao_temporal_spp.argtypes = [P, P, P, I, P, P, P, F, P, P, P]
        L.orc_num_threads.restype = C.c_int
        L.orc_set_num_threads.argtypes = [C.c_int]
        L.orc_shading_create.restype = C.c_void_p
        L.orc_shading_create.argtypes = [P, P, P, P, C.c_size_t, P, C.c_size_t]
        L.orc_shading_destroy.argtypes = [P]
        U = C.c_uint32
        L.orc_ddgi_ray_trace.argtypes = [P, P, P, P, U, F, P, P, P, P, P]
        L.orc_ddgi_probe_update.argtypes = [P, P, P, P, I, I, P]
        L.orc_ddgi_border_update.argtypes = [P, I, P]
        L.orc_ddgi_sample_probe_grid.argtypes = [P, P, P, P, P, F, P]
        L.orc_reflections_ray_trace.argtypes = [P, P, P, F, F, I, I, F, F, P, P, P, P, P, P, P]
        L.orc_reflections_ray_trace_spp.argtypes = [P, P, P, F, F, I, I, F, F, P, I, P, P, P, P, P, P, P, F]
        L.orc_deferred.argtypes = [P, P, P, I, P, P, P, P, P, P]
        L.orc_reflections_temporal.argtypes = [P, P, P, P, P, P, F, F, I, P, P, P]
        L.orc_reflections_atrous.argtypes = [P, P, P, I, I, F, F, F, I, P]
        L.orc_upsample_vec4.argtypes = [P, P, P, P]
        L.orc_rng_sequence.restype = U
        L.orc_rng_sequence.argtypes = [U, U, U, P, I]
        L.orc_gbuffer_render.argtypes = [P, P, P, I, I, P, P, P, P]
        L.orc_taa.argtypes = [I, I, P, I, P, P, P, P, F, F, I, P]
        L.orc_blit_rgba16f.argtypes = [I, I, P, I, P]
        L.orc_taa_jitter.argtypes = [U, I, I, P]
        L.orc_tonemap.argtypes = [I, I, P, I, F, I, P]
        L.orc_path_trace.argtypes = [P, P, I, I, U, U, F, P, P, P, P]
        L.orc_shading_set_textures.argtypes = [P, P, C.c_size_t, P, C.c_size_t, P, P]
        L.orc_fetch_normal.argtypes = [P, P, P, C.c_size_t, I, P]
        L.orc_texture_sample.argtypes = [P, P, C.c_size_t, P]
        L.orc_fetch_material.argtypes = [P, P, P, C.c_size_t, P]
        _lib = L
    return _lib


def p(a):
    return a.ctypes.data_as(C.c_void_p)


class Scene:
    def __init__(self, tri_verts9: np.ndarray, brute=False):
        self.tris = np.ascontiguousarray(tri_verts9, np.float32)
        self.h = lib().orc_scene_create(p(self.tris), self.tris.shape[0], int(brute))

    def set_brute(self, b):
        lib().orc_scene_set_brute(self.h, int(b))

    def trace_any(self, rays):
        rays = np.ascontiguousarray(rays, np.float32)
        out = np.empty(rays.shape[0], np.uint32)
        lib().orc_trace_any(self.h, p(rays), rays.shape[0], p(out))
        return out

    def trace_closest(self, rays):
        rays = np.ascontiguousarray(rays, np.float32)
        n = rays.shape[0]
        t = np.empty(n, np.float32)
        prim = np.empty(n, np.uint32)
        uv = np.empty((n, 2), np.float32)
        lib().orc_trace_closest(self.h, p(rays), n, p(t), p(prim), p(uv))
        return t, prim, uv

    def __del__(self):
        try:
            lib().orc_scene_destroy(self.h)
        except Exception:
            pass


class GBufMips:
    """Host G-buffer with the NEAREST mip chain (oracle statement of g_buffer.cpp:236-244)."""

    def __init__(self, g: "pyhr.GBufferHost", n_mips=3):
        self.levels = [(g.W, g.H, g.gb2, g.gb3, g.depth)]
        for _ in range(1, n_mips):
            W, H, gb2, gb3, d = self.levels[-1]
            w, h = max(W // 2, 1), max(H // 2, 1)
            o2 = np.empty((h, w, 4), np.uint16)
            o3 = np.empty((h, w, 4), np.uint16)
            od = np.empty((h, w), np.float32)
            lib().orc_build_mip(W, H, p(gb2), p(gb3), p(d), p(o2), p(o3), p(od))
            self.levels.append((w, h, o2, o3, od))

    def c(self, mip):
        W, H, gb2, gb3, d = self.levels[mip]
        return orc_gbuf(W, H, p(gb2), p(gb3), p(d))

    def size(self, mip):
        return self.levels[mip][0], self.levels[mip][1]


def zero_gbuf_mips(W, H, n_mips=3):
    return GBufMips(pyhr.GBufferHost(W, H), n_mips)


def _coop_mask(o):
    """keep only the mask rows of this rank's ray-trace share, trash the rest, then let the exchange complete the image"""
    a, b = o.rt_share
    rng = np.random.default_rng(a * 31 + b)
    for sl in (slice(0, a), slice(b, o.mask.shape[0])):
        if o.mask[sl].size:
            o.mask[sl] = rng.integers(0, 2**32, size=o.mask[sl].shape, dtype=np.uint64).astype(np.uint32)
    o.mask[:] = o.mask_exchange(o.mask, a, b)


class ShadowsOracle:
    def __init__(self, W0, H0, scale=0, spp=1):
        self.W0, self.H0, self.scale = W0, H0, scale
        self.W, self.H = W0, H0
        for _ in range(scale):
            self.W, self.H = max(self.W // 2, 1), max(self.H // 2, 1)
        W, H = self.W, self.H
        self.spp = spp  # > 1: SURVEY.md §8d definition (count image instead of the bit mask)
        self.count = np.zeros((H, W), np.uint8)
        self.mask = np.zeros(((H + 3) // 4, (W + 7) // 8), np.uint32)
        self.temporal = np.zeros((H, W, 2), np.uint16)
        self.moments = [np.zeros((H, W, 4), np.uint16), np.zeros((H, W, 4), np.uint16)]
        self.prev_image = np.zeros((H, W, 2), np.uint16)
        self.atrous = [np.zeros((H, W, 2), np.uint16), np.zeros((H, W, 2), np.uint16)]
        self.tile_flags = np.zeros(((H + 7) // 8, (W + 7) // 8), np.uint8)
        self.upsample = np.zeros((H0, W0), np.uint16) if scale else None
        self.first = True
        self.params = pyhr.hr_shadows_params()
        pyhr.load_product  # noqa: B018  (defaults restated here so the oracle does not need the CUDA library)
        P = self.params
        P.bias, P.alpha, P.moments_alpha, P.phi_visibility, P.phi_normal, P.sigma_depth, P.power = 0.5, 0.01, 0.2, 10.0, 32.0, 1.0, 1.2
        P.radius, P.filter_iterations, P.feedback_iteration, P.denoise = 1, 4, 1, 1
        self.final = None
        self.band = None  # (b0, b1): emulate a sharded rank — rows a rank would not compute are overwritten with garbage
        self.halos = (16, 24)  # (denoise, ray trace) rows beyond the band a rank recomputes: hr_shard_halo_rows for the parameters above
        # cooperative ray trace emulation (DESIGN.md §9): this rank traces mask rows [rt_share[0], rt_share[1]) only and
        # mask_exchange(mask, a, b) must return the complete mask (what k_rt_push + the frame ticks do between GPUs)
        self.rt_share, self.mask_exchange = None, None

    def _poison(self, arr, halo, div=1, shift=0):
        """Sharding emulation (tests/test_sharding_cpu.py): keep rows [b0-halo, b1+halo) of a stage output, trash the rest."""
        if self.band is None:
            return
        b0, b1 = self.band
        e0, e1 = max(b0 - halo, 0), min(b1 + halo, self.H)
        if shift:
            e0, e1 = e0 << shift, (arr.shape[0] if e1 >= self.H else e1 << shift)
        e0, e1 = e0 // div, -(-e1 // div)
        rng = np.random.default_rng(e0 * 7919 + e1)
        for sl in (slice(0, e0), slice(e1, arr.shape[0])):
            if arr[sl].size:
                arr[sl] = rng.integers(0, 0x3C00, size=arr[sl].shape, dtype=np.uint32).astype(arr.dtype)

    def render(self, scene: Scene, cur: GBufMips, prev: GBufMips, frame, bn):
        L, P, pp = lib(), self.params, frame.ping_pong
        sobol, sr = bn
        if self.first:
            self.prev_image[:] = 0
            self.moments[1 - pp][:] = 0
            self.first = False
        gc, gp = cur.c(self.scale), prev.c(self.scale)
        if self.spp > 1:
            L.orc_shadows_ray_trace_spp(scene.h, C.byref(gc), C.byref(frame), P.bias, self.spp, p(sobol), p(sr), p(self.count))
            self.final = self.count
            if not P.denoise:
                return
            L.orc_shadows_temporal_spp(C.byref(gc), C.byref(gp), p(self.count), self.spp, p(self.prev_image), p(self.moments[1 - pp]), C.byref(frame),
                                       P.alpha, P.moments_alpha, p(self.temporal), p(self.moments[pp]), p(self.tile_flags))
        else:
            L.orc_shadows_ray_trace(scene.h, C.byref(gc), C.byref(frame), P.bias, p(sobol), p(sr), p(self.mask))
            if self.rt_share is not None:
                _coop_mask(self)
            else:
                self._poison(self.mask, self.halos[1], div=4)
            self.final = self.mask
            if not P.denoise:
                return
            L.orc_shadows_temporal(C.byref(gc), C.byref(gp), p(self.mask), p(self.prev_image), p(self.moments[1 - pp]), C.byref(frame), P.alpha,
                                   P.moments_alpha, p(self.temporal), p(self.moments[pp]), p(self.tile_flags))
        self.cur_moments = self.moments[pp]
        for a in (self.temporal, self.moments[pp], self.tile_flags):
            self._poison(a, self.halos[0], div=8 if a is self.tile_flags else 1)
        ping = False
        src = self.temporal
        for i in range(P.filter_iterations):
            write_idx = int(not ping)
            power = P.power if i == P.filter_iterations - 1 else 0.0
            L.orc_shadows_atrous(C.byref(gc), p(src), p(self.tile_flags), P.radius, 1 << i, P.phi_visibility, P.phi_normal, P.sigma_depth, power,
                                 p(self.atrous[write_idx]))
            self._poison(self.atrous[write_idx], self.halos[0])
            ping = not ping
            if P.feedback_iteration == i:
                self.prev_image[:] = self.atrous[write_idx]
            src = self.atrous[write_idx]
        self.atrous_out = src
        self.final = src
        if self.scale:
            g0 = cur.c(0)
            L.orc_upsample_scalar(C.byref(g0), C.byref(gc), p(src), 2, 0.0, 0.0, p(self.upsample))
            self._poison(self.upsample, 0, shift=self.scale)
            self.final = self.upsample


class AOOracle:
    def __init__(self, W0, H0, scale=1, spp=1):
        self.W0, self.H0, self.scale = W0, H0, scale
        self.W, self.H = W0, H0
        for _ in range(scale):
            self.W, self.H = max(self.W // 2, 1), max(self.H // 2, 1)
        W, H = self.W, self.H
        self.spp = spp
        self.count = np.zeros((H, W), np.uint8)
        self.mask = np.zeros(((H + 3) // 4, (W + 7) // 8), np.uint32)
        self.color = [np.zeros((H, W), np.uint16), np.zeros((H, W), np.uint16)]
        self.length = [np.zeros((H, W), np.uint16), np.zeros((H, W), np.uint16)]
        self.blur = [np.zeros((H, W), np.uint16), np.zeros((H, W), np.uint16)]
        self.tile_flags = np.zeros(((H + 7) // 8, (W + 7) // 8), np.uint8)
        self.upsample = np.zeros((H0, W0), np.uint16) if scale else None
        self.first = True
        self.params = pyhr.hr_ao_params()
        P = self.params
        P.ray_length, P.bias, P.alpha, P.power, P.blur_radius, P.denoise = 7.0, 0.3, 0.01, 1.2, 4, 1
        self.final = None
        self.band = None

    _poison = ShadowsOracle._poison

    def render(self, scene: Scene, cur: GBufMips, prev: GBufMips, frame, bn):
        L, P, pp = lib(), self.params, frame.ping_pong
        sobol, sr = bn
        if self.first:
            self.color[1 - pp][:] = 0
            self.length[1 - pp][:] = 0
            self.first = False
        gc, gp = cur.c(self.scale), prev.c(self.scale)
        if self.spp > 1:
            L.orc_ao_ray_trace_spp(scene.h, C.byref(gc), C.byref(frame), P.ray_length, P.bias, self.spp, p(sobol), p(sr), p(self.count))
            self.final = self.count
            if not P.denoise:
                return
            L.orc_ao_temporal_spp(C.byref(gc), C.byref(gp), p(self.count), self.spp, p(self.color[1 - pp]), p(self.length[1 - pp]), C.byref(frame),
                                  P.alpha, p(self.color[pp]), p(self.length[pp]), p(self.tile_flags))
        else:
            L.orc_ao_ray_trace(scene.h, C.byref(gc), C.byref(frame), P.ray_length, P.bias, p(sobol), p(sr), p(self.mask))
            if getattr(self, "rt_share", None) is not None:
                _coop_mask(self)
            else:
                self._poison(self.mask, 24, div=4)
            self.final = self.mask
            if not P.denoise:
                return
            L.orc_ao_temporal(C.byref(gc), C.byref(gp), p(self.mask), p(self.color[1 - pp]), p(self.length[1 - pp]), C.byref(frame), P.alpha,
                              p(self.color[pp]), p(self.length[pp]), p(self.tile_flags))
        self.temporal = self.color[pp]
        self.cur_length = self.length[pp]
        for a in (self.color[pp], self.length[pp], self.tile_flags):
            self._poison(a, 16, div=8 if a is self.tile_flags else 1)
        zbp = np.array(frame.z_buffer_params[:], np.float32)
        L.orc_ao_bilateral_blur(C.byref(gc), p(self.color[pp]), p(self.tile_flags), p(zbp), 1, 0, P.blur_radius, p(self.blur[0]))
        self._poison(self.blur[0], 16)
        L.orc_ao_bilateral_blur(C.byref(gc), p(self.blur[0]), p(self.tile_flags), p(zbp), 0, 1, P.blur_radius, p(self.blur[1]))
        self._poison(self.blur[1], 8)
        self.final = self.blur[1]
        if self.scale:
            g0 = cur.c(0)
            L.orc_upsample_scalar(C.byref(g0), C.byref(gc), p(self.blur[1]), 1, 1.0, P.power, p(self.upsample))
            self._poison(self.upsample, 0, shift=self.scale)
            self.final = self.upsample


def h2f(a):
    """uint16 half bits -> float32"""
    return np.ascontiguousarray(a).view(np.float16).astype(np.float32)


class ShadingScene:
    """oracle-side scene with shading data (positions, vertex normals, materials) in primitive order"""

    def __init__(self, synth_scene, brute=False):
        tri, _ = synth_scene.world_triangles()
        nrm, mat = synth_scene.world_normals()
        self.scene = Scene(tri, brute)
        self.tri, self.nrm, self.mat = tri, nrm, mat
        self.synth = synth_scene
        mats = synth_scene.materials_array()
        self.h = lib().orc_shading_create(self.scene.h, p(tri), p(nrm), p(mat), tri.shape[0], C.cast(mats, C.c_void_p), synth_scene.n_materials)

    def set_textures(self, textures, bindings, vuv, vtb=None):
        """hr_scene_set_textures on the oracle's scene: textures = [(uint8 array, srgb)], bindings = [dict] per material (keys of
        hr_material_textures), vuv = (n_tris, 6) texture coordinates per primitive corner"""
        self._tex_keep = [np.ascontiguousarray(a, np.uint8) for a, _ in textures]
        tx = (pyhr.hr_texture * max(1, len(textures)))()
        for i, (a, (_, srgb)) in enumerate(zip(self._tex_keep, textures)):
            tx[i] = pyhr.hr_texture(a.shape[1], a.shape[0], 1 if a.ndim == 2 else a.shape[2], int(bool(srgb)), a.ctypes.data)
        bd = (pyhr.hr_material_textures * max(1, len(bindings)))()
        for i, b in enumerate(bindings):
            bd[i] = pyhr.hr_material_textures(b.get("albedo", -1), b.get("normal", -1), b.get("roughness", -1), b.get("roughness_channel", 0), b.get("metallic", -1),
                                              b.get("metallic_channel", 0), b.get("emissive", -1))
        vuv = np.ascontiguousarray(vuv, np.float32)
        assert not textures or vuv.shape == (self.tri.shape[0], 6)
        if vtb is not None:
            vtb = np.ascontiguousarray(vtb, np.float32)
            assert vtb.shape == (self.tri.shape[0], 18)
        lib().orc_shading_set_textures(self.h, tx, len(textures), bd, len(bindings), p(vuv), p(vtb) if vtb is not None else None)

    def __del__(self):
        try:
            lib().orc_shading_destroy(self.h)
        except Exception:
            pass


def fetch_material(ss: "ShadingScene", prim, bary_uv):
    """fetch_surface's albedo rgb / roughness / metallic at hits (primitive, u, v): (n, 5) float32"""
    prim = np.ascontiguousarray(prim, np.uint32)
    uv = np.ascontiguousarray(bary_uv, np.float32).reshape(-1, 2)
    out = np.empty((len(prim), 5), np.float32)
    lib().orc_fetch_material(ss.h, p(prim), p(uv), len(prim), p(out))
    return out


def fetch_normal(ss: "ShadingScene", prim, bary_uv, hit_shader=True):
    """the shading normal fetch_normal returns at hits (primitive, u, v): (n, 3) float32; hit_shader: the rchit call (tangent as bitangent)"""
    prim = np.ascontiguousarray(prim, np.uint32)
    uv = np.ascontiguousarray(bary_uv, np.float32).reshape(-1, 2)
    out = np.empty((len(prim), 3), np.float32)
    lib().orc_fetch_normal(ss.h, p(prim), p(uv), len(prim), int(hit_shader), p(out))
    return out


def texture_sample(img, srgb, uv):
    """texture(sampler2D over img (uint8 (H, W[, C])), uv) at mip 0, bilinear, REPEAT: (n, 4) float32"""
    a = np.ascontiguousarray(img, np.uint8)
    t = pyhr.hr_texture(a.shape[1], a.shape[0], 1 if a.ndim == 2 else a.shape[2], int(bool(srgb)), a.ctypes.data)
    uv = np.ascontiguousarray(uv, np.float32).reshape(-1, 2)
    out = np.empty((len(uv), 4), np.float32)
    lib().orc_texture_sample(C.byref(t), p(uv), len(uv), p(out))
    return out


def gbuffer_render(ss: "ShadingScene", frame, W, H, out=None):
    """oracle statement of the device G-buffer producer (oracle/orc_gbuffer.cpp) -> pyhr.GBufferHost"""
    g = out if out is not None else pyhr.GBufferHost(W, H)
    _, inst = ss.synth.world_triangles()
    inst = np.ascontiguousarray(inst, np.uint32)
    lib().orc_gbuffer_render(ss.h, p(inst), C.byref(frame), W, H, p(g.gb1), p(g.gb2), p(g.gb3), p(g.depth))
    return g


def ddgi_uniforms_from(params, bounds_min, bounds_max):
    """initialize_probe_grid + update_properties_ubo (ddgi.cpp:150-169, :738-763)"""
    u = pyhr.hr_ddgi_uniforms()
    for a in range(3):
        ln = np.float32(bounds_max[a]) - np.float32(bounds_min[a])
        u.probe_counts[a] = int(np.float32(ln) / np.float32(params.probe_distance)) + 2
        u.grid_start_position[a] = float(bounds_min[a])
        u.grid_step[a] = params.probe_distance
    cx, cy, cz = u.probe_counts[0], u.probe_counts[1], u.probe_counts[2]
    u.max_distance = params.probe_distance * 1.5
    u.depth_sharpness, u.hysteresis, u.normal_bias = params.depth_sharpness, params.hysteresis, params.normal_bias
    u.energy_preservation = params.recursive_energy_preservation
    u.irradiance_probe_side_length, u.depth_probe_side_length = params.irradiance_oct_size, params.depth_oct_size
    u.irradiance_texture_width = (params.irradiance_oct_size + 2) * cx * cy + 2
    u.irradiance_texture_height = (params.irradiance_oct_size + 2) * cz + 2
    u.depth_texture_width = (params.depth_oct_size + 2) * cx * cy + 2
    u.depth_texture_height = (params.depth_oct_size + 2) * cz + 2
    u.rays_per_probe, u.visibility_test = params.rays_per_probe, params.visibility_test
    return u


class DDGIOracle:
    """DDGI::render, src/ddgi.cpp:89-104"""

    def __init__(self, W0, H0, scale, params, bounds_min, bounds_max):
        self.W, self.H, self.scale = W0 >> scale, H0 >> scale, scale
        self.params = params
        self.u = ddgi_uniforms_from(params, bounds_min, bounds_max)
        u = self.u
        self.total = u.probe_counts[0] * u.probe_counts[1] * u.probe_counts[2]
        self.radiance = np.zeros((self.total, u.rays_per_probe, 4), np.uint16)
        self.dirdepth = np.zeros((self.total, u.rays_per_probe, 4), np.uint16)
        self.irr = [np.zeros((u.irradiance_texture_height, u.irradiance_texture_width, 4), np.uint16) for _ in range(2)]
        self.dep = [np.zeros((u.depth_texture_height, u.depth_texture_width, 2), np.uint16) for _ in range(2)]
        self.sample = np.zeros((self.H, self.W, 4), np.uint16)
        self.mp, self.first = 0, True

    def render(self, ss: ShadingScene, cur: GBufMips, frame, rot16):
        L, P, u, mp = lib(), self.params, self.u, self.mp
        sky = np.array(P.sky_color[:], np.float32)
        rot = np.ascontiguousarray(rot16, np.float32)
        inf = 1 if (P.infinite_bounces and not self.first) else 0
        L.orc_ddgi_ray_trace(ss.h, C.byref(u), C.byref(frame), p(rot), inf, P.infinite_bounce_intensity, p(sky), p(self.irr[1 - mp]), p(self.dep[1 - mp]),
                             p(self.radiance), p(self.dirdepth))
        ff = 1 if self.first else 0
        L.orc_ddgi_probe_update(C.byref(u), p(self.radiance), p(self.dirdepth), p(self.irr[1 - mp]), ff, 0, p(self.irr[mp]))
        L.orc_ddgi_probe_update(C.byref(u), p(self.radiance), p(self.dirdepth), p(self.dep[1 - mp]), ff, 1, p(self.dep[mp]))
        L.orc_ddgi_border_update(C.byref(u), 0, p(self.irr[mp]))
        L.orc_ddgi_border_update(C.byref(u), 1, p(self.dep[mp]))
        gc = cur.c(self.scale)
        L.orc_ddgi_sample_probe_grid(C.byref(gc), C.byref(frame), C.byref(u), p(self.irr[mp]), p(self.dep[mp]), P.gi_intensity, p(self.sample))
        self.cur_irr, self.cur_dep = self.irr[mp], self.dep[mp]
        self.first = False
        self.mp = 1 - mp


class ReflectionsOracle:
    """RayTracedReflections::render, src/ray_traced_reflections.cpp:107-123"""

    def __init__(self, W0, H0, scale, params):
        self.W0, self.H0, self.scale = W0, H0, scale
        self.W, self.H = W0 >> scale, H0 >> scale
        W, H = self.W, self.H
        self.params = params
        self.rt = np.zeros((H, W, 4), np.uint16)
        self.temporal = [np.zeros((H, W, 4), np.uint16) for _ in range(2)]
        self.moments = [np.zeros((H, W, 4), np.uint16) for _ in range(2)]
        self.prev_image = np.zeros((H, W, 4), np.uint16)
        self.atrous = [np.zeros((H, W, 4), np.uint16) for _ in range(2)]
        self.tile_flags = np.zeros(((H + 7) // 8, (W + 7) // 8), np.uint8)
        self.upsample = np.zeros((H0, W0, 4), np.uint16) if scale else None
        self.first = True
        self.final = None
        # sharding emulation (tests/test_sharding_cpu.py, DESIGN.md §9): band = (b0, b1) rows this rank owns, halos = (denoise, ray trace)
        # rows beyond it that it recomputes (hr_shard_halo_rows); rt_chunks = (rank, world): this rank traces only the 8-row chunks
        # c % world == rank and rt_exchange(image) must return the complete ray-trace image (what k_rt_push_chunks + the ticks do)
        self.band, self.halos, self.rt_chunks, self.rt_exchange = None, (0, 0), None, None

    _poison = ShadowsOracle._poison

    def render(self, ss: ShadingScene, cur: GBufMips, prev: GBufMips, frame, bn, ddgi: DDGIOracle = None):
        L, P, pp = lib(), self.params, frame.ping_pong
        sobol, sr = bn
        if self.first:
            self.prev_image[:] = 0
            self.moments[1 - pp][:] = 0
            self.temporal[1 - pp][:] = 0
        have_gi = ddgi is not None
        sample_gi = 1 if (P.sample_gi and have_gi and not self.first) else 0
        approx = 1 if (P.approximate_with_ddgi and have_gi and not self.first) else 0
        sky = np.array(P.sky_color[:], np.float32)
        gc, gp = cur.c(self.scale), prev.c(self.scale)
        # reflections read the atlas DDGI wrote this frame (ddgi.cpp:100-103,135-138)
        up = C.byref(ddgi.u) if have_gi else None
        irr = p(ddgi.cur_irr) if have_gi else None
        dep = p(ddgi.cur_dep) if have_gi else None
        spp = max(1, int(getattr(P, "spp", 1)))
        lut = getattr(self, "brdf_lut", None)  # 512 x 512 x 2 uint16 (RG16F) or None: IBL specular term of the hit shading
        if spp > 1 or lut is not None:
            L.orc_reflections_ray_trace_spp(ss.h, C.byref(gc), C.byref(frame), P.bias, P.trim, sample_gi, approx, P.gi_intensity, P.rough_ddgi_intensity, p(sky), spp,
                                            p(sobol), p(sr), up, irr, dep, p(self.rt), p(lut) if lut is not None else None, P.ibl_indirect_specular_intensity)
        else:
            L.orc_reflections_ray_trace(ss.h, C.byref(gc), C.byref(frame), P.bias, P.trim, sample_gi, approx, P.gi_intensity, P.rough_ddgi_intensity, p(sky), p(sobol), p(sr),
                                        up, irr, dep, p(self.rt))
        if self.rt_chunks is not None:
            rank, world = self.rt_chunks
            rng = np.random.default_rng(4242 + rank)
            for c in range((self.H + 7) // 8):
                if c % world != rank:  # not traced by this rank
                    rows = self.rt[c * 8:c * 8 + 8]
                    rows[:] = rng.integers(0, 0x3C00, size=rows.shape, dtype=np.uint32).astype(np.uint16)
            self.rt[:] = self.rt_exchange(self.rt)
        self._poison(self.rt, self.halos[1] if P.denoise else 0)
        self.final = self.rt
        self.first = False
        if not P.denoise:
            return
        hist = self.prev_image if P.blur_as_input else self.temporal[1 - pp]
        L.orc_reflections_temporal(C.byref(gc), C.byref(gp), p(self.rt), p(hist), p(self.moments[1 - pp]), C.byref(frame), P.alpha, P.moments_alpha, approx,
                                   p(self.temporal[pp]), p(self.moments[pp]), p(self.tile_flags))
        self.cur_temporal, self.cur_moments = self.temporal[pp], self.moments[pp]
        for a in (self.temporal[pp], self.moments[pp], self.tile_flags):
            self._poison(a, self.halos[0], div=8 if a is self.tile_flags else 1)
        src, toggle = self.temporal[pp], 1
        for i in range(P.filter_iterations):
            dst = self.atrous[toggle]
            L.orc_reflections_atrous(C.byref(gc), p(src), p(self.tile_flags), P.radius, 1 << i, P.phi_color, P.phi_normal, P.sigma_depth, approx, p(dst))
            self._poison(dst, self.halos[0])
            if P.blur_as_input and i == P.feedback_iteration:
                self.prev_image[:] = dst
            src, toggle = dst, 1 - toggle
        self.atrous_out = src
        self.final = src
        if self.scale:
            g0 = cur.c(0)
            L.orc_upsample_vec4(C.byref(g0), C.byref(gc), p(src), p(self.upsample))
            self._poison(self.upsample, 0, shift=self.scale)
            self.final = self.upsample


class orc_gbuf_full(C.Structure):
    _fields_ = [("W", C.c_int32), ("H", C.c_int32), ("gb1", C.c_void_p), ("gb2", C.c_void_p), ("gb3", C.c_void_p), ("depth", C.c_void_p)]


def deferred(g: "pyhr.GBufferHost", frame, shadow=None, ao=None, reflections=None, gi=None, env=(0.0, 0.0, 0.0), brdf_lut=None):
    """oracle statement of the deferred shading combine (oracle/orc_deferred.cpp); inputs are full-resolution uint16 (half) images"""
    gf = orc_gbuf_full(g.W, g.H, p(g.gb1), p(g.gb2), p(g.gb3), p(g.depth))
    out = np.zeros((g.H, g.W, 4), np.uint16)
    envv = np.array(env, np.float32)
    ch = 0 if shadow is None else (shadow.shape[2] if shadow.ndim == 3 else 1)
    arrs = [np.ascontiguousarray(a) if a is not None else None for a in (shadow, ao, reflections, gi)]
    lib().orc_deferred(C.byref(gf), C.byref(frame), p(arrs[0]) if arrs[0] is not None else None, ch, p(arrs[1]) if arrs[1] is not None else None,
                       p(arrs[2]) if arrs[2] is not None else None, p(arrs[3]) if arrs[3] is not None else None, p(envv),
                       p(brdf_lut) if brdf_lut is not None else None, p(out))
    return out


# ---------------------------------------------------------------------------------------------- post-processing (oracle/orc_post.cpp)
def _channels(img):
    return 1 if img.ndim == 2 else img.shape[2]


def taa_jitter(num_frames, W, H):
    """TemporalAA::update (temporal_aa.cpp:66-81): jitter of frame num_frames"""
    out = np.zeros(2, np.float32)
    lib().orc_taa_jitter(num_frames, W, H, p(out))
    return out


def blit_rgba16f(src):
    """vkCmdBlitImage into an RGBA16F image: (H, W[, C]) uint16 halves -> (H, W, 4)"""
    src = np.ascontiguousarray(src, np.uint16)
    H, W = src.shape[:2]
    out = np.empty((H, W, 4), np.uint16)
    lib().orc_blit_rgba16f(W, H, p(src), _channels(src), p(out))
    return out


def taa(cur, prev, depth, gb2, jitter_xy, feedback_min=0.88, feedback_max=0.97, sharpen=1):
    """taa.comp over the whole image: cur (H, W[, C]) halves, prev (H, W, 4) halves, depth (H, W) f32, gb2 (H, W, 4) halves"""
    cur, prev, gb2 = (np.ascontiguousarray(a, np.uint16) for a in (cur, prev, gb2))
    depth = np.ascontiguousarray(depth, np.float32)
    H, W = cur.shape[:2]
    j = np.ascontiguousarray(jitter_xy, np.float32)
    out = np.empty((H, W, 4), np.uint16)
    lib().orc_taa(W, H, p(cur), _channels(cur), p(prev), p(depth), p(gb2), p(j), feedback_min, feedback_max, int(sharpen), p(out))
    return out


def tonemap(src, exposure=1.0, single_channel=0):
    src = np.ascontiguousarray(src, np.uint16)
    H, W = src.shape[:2]
    out = np.empty((H, W, 4), np.uint8)
    lib().orc_tonemap(W, H, p(src), _channels(src), exposure, int(single_channel), p(out))
    return out


class TAAOracle:
    """TemporalAA::render (temporal_aa.cpp:83-172) host sequencing on the oracle: two RGBA16F images indexed by ping_pong, the reset
    blit (reset_every_frame = the reference as written, see hr_taa_params)"""

    def __init__(self, W, H, feedback_min=0.88, feedback_max=0.97, sharpen=1, reset_every_frame=1):
        self.img = [np.zeros((H, W, 4), np.uint16), np.zeros((H, W, 4), np.uint16)]
        self.first = True
        self.fmin, self.fmax, self.sharpen, self.reset_every_frame = feedback_min, feedback_max, sharpen, reset_every_frame

    def render(self, frame, cur, depth, gb2):
        w, r = frame.ping_pong, 1 - frame.ping_pong
        if self.first or self.reset_every_frame:
            self.img[r] = blit_rgba16f(cur)
            self.first = False
        self.img[w] = taa(cur, self.img[r], depth, gb2, frame.ubo.current_prev_jitter[0:2], self.fmin, self.fmax, self.sharpen)
        return self.img[w]


# ---------------------------------------------------------------------------------------------- ground-truth path tracer (oracle/orc_path_trace.cpp)
class PathTracerOracle:
    """GroundTruthPathTracer::render host sequencing (ground_truth_path_tracer.cpp:44-113): frame counter, two images, ping-pong"""

    def __init__(self, W, H, max_ray_bounces=2, roughness_multiplier=1.0, sky=(0.0, 0.0, 0.0)):
        self.W, self.H = W, H
        self.img = [np.zeros((H, W, 4), np.uint16), np.zeros((H, W, 4), np.uint16)]
        self.prim = np.full((H, W), 0xFFFFFFFF, np.uint32)
        self.frame_idx, self.ping_pong = 0, 0
        self.max_ray_bounces, self.roughness_multiplier, self.sky = max_ray_bounces, roughness_multiplier, np.asarray(sky, np.float32)

    def restart_accumulation(self):
        self.frame_idx = 0

    def render(self, ss: "ShadingScene", frame):
        if self.frame_idx == 0:
            self.ping_pong = 0
        r, w = self.ping_pong, 1 - self.ping_pong
        lib().orc_path_trace(ss.h, C.byref(frame), self.W, self.H, self.frame_idx, self.max_ray_bounces, self.roughness_multiplier, p(self.sky), p(self.img[r]),
                             p(self.img[w]), p(self.prim))
        self.frame_idx += 1
        self.ping_pong = 1 - self.ping_pong
        self.final = self.img[w]
        return self.final
