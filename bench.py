#!/usr/bin/env python
"""bench.py — denoised frames/s of the ray-trace + SVGF hot path on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config {1,2,3,4,5}] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one frame of the configuration's passes.  --config picks one of BASELINE.json's five configurations as
SURVEY.md §8d makes them concrete; the default is the largest single-GPU one, config 3:

  3  3840x2160, 1 spp reflections at FULL resolution + SVGF (K12 ray trace + hit shading, K14 temporal, 4x K16 a-trous),
     262 144-triangle arcade, roughness per mesh in {0.02, 0.2, 0.5, 0.9}, no DDGI (approximate_with_ddgi = sample_gi = 0)
  2  1920x1080 shadows (full-res) + AO (reference default half-res), full denoise chains
  1  256x256 analytic ground plane, single-triangle BVH, 1 spp shadows, no denoise
  4  3840x2160 shadows + AO + DDGI (4096 probes x 256 rays) + reflections, 2 spp
  5  7680x4320, 4 spp, ~1 M triangles, all passes

What is measured (all through the C ABI, CUDA events on the launch stream, W >= 3 warm-up steps + history warm-up, K timed
steps between barrier + synchronize, max over ranks):
  value     frames/s with the G-buffer resident in HBM (static camera, steady state: history saturated; the blue-noise sample
            index advances every frame so the traced rays change every frame).  N > 1: the frame is split into row bands and the
            final output is all-gathered to every rank INSIDE the timed region (value_distributed = without the gather)
  pan       the same passes over a 40-frame lateral camera pan (0.05 units / frame): the G-buffer is produced on the device
            every frame by hr_gbuffer_render (its time is reported separately), reprojection follows real motion vectors
  e2e       frames/s from HOST inputs to HOST outputs, every step: the host builds the 496-byte hr_frame (camera, light,
            matrices) -> hr_gbuffer_render on the device (SURVEY.md §8 f1: the G-buffer is produced where the reference
            produces it, on the GPU) -> passes -> the denoised outputs are copied to pinned host memory (staged through one
            device buffer so the PCIe copy of frame N overlaps frame N+1).  e2e.host_gbuffer_value is the older mode that
            uploads a host G-buffer every frame (GB2 + GB3 + depth, 20 B/px over PCIe)
  roofline  the configuration's a-trous kernel (K16 reflections for configs 3-5, K5 shadows for 1-2): ALGORITHMIC bytes
            (SURVEY.md §8d: 36 resp. 24 B/px/iteration) of the pixels the launch PROCESSED — 8x8 tiles on the denoise list
            count fully, copy / zero-filled tiles count only their real bytes — / the average CUDA-event duration of a launch.
            frac_contract is the whole-frame 36 (24) B/px figure for comparison.  k5_dense: the shadows a-trous on a view
            where >= 95 % of the tiles are on the denoise list (no help from sparsity)
  post_passes   (N = 1, informational, own process) deferred combine -> TAA -> tone map and the ground-truth path tracer at the bench
            resolution: ms per launch, roofline fractions on their algorithmic bytes (36 / 12 B/px), Mrays/s of the path tracer
  cpu_baseline / --impl reference   the CPU oracle (a port: the reference has no CPU path and cannot be built here),
            OpenMP over all host threads (set explicitly), best of 5 frames on a 1/16-area render of the same workload
            (same scene and passes), stated as frames/s of that SAMPLE and extrapolated x16 in `value`

Inputs (G-buffer 199 MB + history / intermediates > 300 MB per 4K frame) exceed the 126 MB L2: "inputs_larger_than_l2".
"""
import argparse
import ctypes as C
import glob
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "hybrid-rendering_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

CAM_POS, CAM_TGT = (0.0, 9.0, -4.0), (2.0, 7.0, 60.0)  # looking down the arcade's nave
LIGHT_ROT_X = 25.0
DENSE_CAM = ((0.0, 18.0, 10.0), (0.0, 0.0, 0.0))        # shadows-test scene from above: no sky, > 95 % of the tiles lit
SKY = (0.3, 0.4, 0.6)
PAN_STEP = 0.05

CONFIGS = {
    1: dict(W=256, H=256, tris=1, passes=["shadows"], spp=1, denoise=False, scene="single_triangle",
            name="256x256 analytic ground plane + single-triangle BVH, 1 spp shadows, no denoise"),
    2: dict(W=1920, H=1080, tris=262144, passes=["shadows", "ao"], spp=1, name="1920x1080 1 spp shadows(full-res)+AO(half-res) full SVGF, arcade 262144 tris"),
    3: dict(W=3840, H=2160, tris=262144, passes=["reflections"], spp=1, refl_scale=0,
            name="3840x2160 1 spp reflections(full-res)+SVGF (K12,K14,4xK16), arcade 262144 tris, no DDGI"),
    4: dict(W=3840, H=2160, tris=262144, passes=["shadows", "ao", "ddgi", "reflections"], spp=2, refl_scale=1,
            name="3840x2160 2 spp shadows+AO(half)+DDGI(4096 probes x 256 rays)+reflections(half), arcade 262144 tris"),
    5: dict(W=7680, H=4320, tris=1000000, passes=["shadows", "ao", "ddgi", "reflections"], spp=4, refl_scale=1,
            name="7680x4320 4 spp shadows+AO(half)+DDGI+reflections(half), arcade ~1M tris"),
}
ATROUS_BYTES = {"reflections": (36.0, 16.0), "shadows": (24.0, 4.0)}  # (B/px on the denoise list, B/px of a copy / zero-filled tile)


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def read_traffic(kernel_key):
    """DRAM bytes per launch of the roofline kernel from the newest committed ncu summary (profiles/*_traffic.json)."""
    best = None
    for p in sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json"))):
        try:
            d = json.load(open(p))
        except Exception:
            continue
        if kernel_key in d:
            best = (d[kernel_key], os.path.relpath(p, ROOT), d.get("_source"))
    return best


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.stop_flag = index, [], set(), None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        self.stop_flag = True
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# ---------------------------------------------------------------------------------------------------------------- CPU arm
def oracle_fps(cfg, scale_div=None, frames=5):
    """The CPU oracle on a 1/scale_div^2-area render of the configuration (same scene, passes, parameters): best of `frames`
    individually timed steady-state frames with every host thread.  Returns a dict for `cpu_baseline`."""
    import oracle as O
    import pyhr
    n_thr = os.cpu_count() or 1
    O.lib().orc_set_num_threads(n_thr)
    W, H = cfg["W"], cfg["H"]
    scale_div = scale_div or (4 if W > 4000 else 2)  # bounded sample: 1/4 area (1/16 at 8K), ~10-30 s of CPU work on a many-core host
    sw, shh = (W // scale_div, H // scale_div) if W > 512 else (W, H)
    extrap = (W * H) / float(sw * shh)
    light = pyhr.default_light(rot_x_deg=LIGHT_ROT_X)
    bn = pyhr.blue_noise()
    spp = cfg.get("spp", 1)
    if cfg.get("scene") == "single_triangle":
        sc, gsc = pyhr.SynthScene(pyhr.SCENE_SINGLE_TRIANGLE), pyhr.SynthScene(pyhr.SCENE_GROUND_PLANE)
        cam, tgt = (0.0, 8.0, 20.0), (0.0, 0.0, 0.0)
        light = pyhr.default_light()
    else:
        sc = gsc = pyhr.SynthScene(pyhr.SCENE_ARCADE, cfg["tris"])
        cam, tgt = CAM_POS, CAM_TGT
    ss = O.ShadingScene(sc, brute=sc.n_tris <= 64)
    osc = ss.scene
    f = pyhr.make_frame(cam, tgt, sw, shh, light=light)
    f = pyhr.make_frame(cam, tgt, sw, shh, prev=f, num_frames=1, light=light)
    g = O.GBufMips(pyhr.write_gbuffer(gsc, f, sw, shh))
    passes = {}
    if "shadows" in cfg["passes"]:
        passes["shadows"] = O.ShadowsOracle(sw, shh, 0, spp=spp)
        passes["shadows"].params.denoise = 1 if cfg.get("denoise", True) else 0
    if "ao" in cfg["passes"]:
        passes["ao"] = O.AOOracle(sw, shh, 1, spp=spp)
    if "ddgi" in cfg["passes"]:
        dp = pyhr.hr_ddgi_params()
        pyhr.load_product().hr_ddgi_default_params(C.byref(dp)) if os.path.exists(pyhr.LIB_PRODUCT) else None
        dp.infinite_bounces, dp.infinite_bounce_intensity, dp.rays_per_probe, dp.visibility_test = 1, 1.7, 256, 1
        dp.recursive_energy_preservation, dp.irradiance_oct_size, dp.depth_oct_size, dp.hysteresis, dp.depth_sharpness, dp.gi_intensity = 0.85, 8, 16, 0.98, 50.0, 1.0
        dp.probe_distance, dp.normal_bias = 4.2, 0.5
        dp.sky_color[0], dp.sky_color[1], dp.sky_color[2] = SKY
        mn, mx = sc.bounds()
        passes["ddgi"] = O.DDGIOracle(sw, shh, 0, dp, mn, mx)
    if "reflections" in cfg["passes"]:
        rp = refl_params(cfg)
        passes["reflections"] = O.ReflectionsOracle(sw, shh, cfg.get("refl_scale", 1), rp)
    rng = np.random.default_rng(1234)

    def one(fr):
        if "shadows" in passes:
            passes["shadows"].render(osc, g, g, fr, bn)
        if "ao" in passes:
            passes["ao"].render(osc, g, g, fr, bn)
        if "ddgi" in passes:
            ax = rng.uniform(-1, 1, 3)
            passes["ddgi"].render(ss, g, fr, pyhr.rotation_matrix(float(rng.uniform(0, 2 * np.pi)), ax / np.linalg.norm(ax)))
        if "reflections" in passes:
            passes["reflections"].render(ss, g, g, fr, bn, passes.get("ddgi"))

    one(f)  # warm-up, leaves valid history
    times = []
    t_all = time.perf_counter()
    for i in range(frames):
        f = pyhr.make_frame(cam, tgt, sw, shh, prev=f, num_frames=2 + i, light=light)
        t0 = time.perf_counter()
        one(f)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > 120.0:
            break
    best = min(times)
    return {"value": 1.0 / (best * extrap), "unit": "frames/s", "cores": int(O.lib().orc_num_threads()), "kind": "port", "cpu_model": cpu_model(),
            "sample": f"{sw}x{shh} render ({'1/%d' % int(round(extrap)) if extrap > 1 else 'full'} area) of the same scene and passes, best of {len(times)} frames "
                      f"(each {', '.join('%.2f' % t for t in times)} s), sample rate {1.0 / best:.3f} frames/s" + (f", extrapolated x{extrap:.0f}" if extrap > 1 else ""),
            "sample_frames_per_s": 1.0 / best, "extrapolation": extrap}


def refl_params(cfg):
    import pyhr
    rp = pyhr.hr_reflections_params()
    rp.bias, rp.trim, rp.gi_intensity, rp.rough_ddgi_intensity, rp.ibl_indirect_specular_intensity = 0.5, 0.8, 0.5, 0.5, 0.05
    rp.alpha, rp.moments_alpha, rp.blur_as_input, rp.phi_color, rp.phi_normal, rp.sigma_depth = 0.01, 0.2, 0, 10.0, 32.0, 1.0
    rp.radius, rp.filter_iterations, rp.feedback_iteration, rp.denoise = 1, 4, 1, 1
    with_ddgi = "ddgi" in cfg["passes"]
    rp.sample_gi, rp.approximate_with_ddgi = (1, 1) if with_ddgi else (0, 0)
    rp.sky_color[0], rp.sky_color[1], rp.sky_color[2] = SKY
    return rp


# ---------------------------------------------------------------------------------------------------------------- GPU rig
class Rig:
    """The configuration's passes on one context, in the reference's frame order (main.cpp:49-129: shadows, AO, DDGI, reflections)."""

    def __init__(self, pyhr, ctx, cfg, W, H):
        self.pyhr, self.ctx, self.cfg = pyhr, ctx, cfg
        self.passes = {}
        spp = cfg.get("spp", 1)
        if "shadows" in cfg["passes"]:
            p = pyhr.Pass(ctx, "shadows", W, H, 0)
            p.params.denoise = 1 if cfg.get("denoise", True) else 0
            p.params.spp = spp
            self.passes["shadows"] = p
        if "ao" in cfg["passes"]:
            p = pyhr.Pass(ctx, "ao", W, H, cfg.get("ao_scale", 1))
            p.params.spp = spp
            self.passes["ao"] = p
        if "ddgi" in cfg["passes"]:
            p = pyhr.DDGIPass(ctx, W, H, 0)
            p.params.probe_distance, p.params.normal_bias = 4.2, 0.5  # arcade bounds 60 x 28.6 x 128 => 16 x 8 x 32 = 4096 probes
            p.params.sky_color[0], p.params.sky_color[1], p.params.sky_color[2] = SKY
            self.passes["ddgi"] = p
        if "reflections" in cfg["passes"]:
            p = pyhr.ReflectionsPass(ctx, W, H, cfg.get("refl_scale", 1))
            src = refl_params(cfg)
            for name, _ in src._fields_:
                if name != "sky_color":
                    setattr(p.params, name, getattr(src, name))
            for k in range(3):
                p.params.sky_color[k] = SKY[k]
            if hasattr(p.params, "spp"):
                p.params.spp = spp
            self.passes["reflections"] = p
        self.rng = np.random.default_rng(1234)
        self.outputs = [p for k, p in self.passes.items()]

    def render(self, f, stream):
        P = self.passes
        if "shadows" in P:
            P["shadows"].render(f, stream)
        if "ao" in P:
            P["ao"].render(f, stream)
        if "ddgi" in P:
            ax = self.rng.uniform(-1, 1, 3)
            P["ddgi"].render(f, self.pyhr.rotation_matrix(float(self.rng.uniform(0, 2 * np.pi)), ax / np.linalg.norm(ax)), stream)
        if "reflections" in P:
            P["reflections"].render(f, P.get("ddgi"), stream)

    def stage_times(self):
        return {k: dict(p.stage_times()) for k, p in self.passes.items()}

    def stats(self, stream):
        return {k: p.stats(stream) for k, p in self.passes.items()}

    def reset(self):
        self.rng = np.random.default_rng(1234)
        for p in self.passes.values():
            p.reset_history()

    def destroy(self):
        for p in self.passes.values():
            p.destroy()


def texel_bytes(img):
    return {1: 4, 2: 2, 3: 4, 4: 8, 5: 1}[img.format]


DUMP_BYTES = 64 * 10**6  # --dump-outputs: all files together stay below this


def dump_outputs(out_dir, images, seed=0):
    """Writes every image as out_dir/<name>.npy: float32 (float64 for 32-bit integer images), shape (H, W[, C]).  An image larger than
    its share of DUMP_BYTES is written as a fixed sample of its pixels drawn with `seed`: (n, C), the pixels in row-major order, so two
    builds given the same arguments write the same pixels."""
    os.makedirs(out_dir, exist_ok=True)
    share = (DUMP_BYTES - 4096 * len(images)) // max(1, len(images))  # 4096: room for each .npy header
    for name, a in images.items():
        a = a.astype(np.float64 if a.dtype.kind in "iu" and a.dtype.itemsize == 4 else np.float32)
        if a.nbytes > share:
            px = a.reshape(a.shape[0] * a.shape[1], -1)
            n = share // (px.shape[1] * px.itemsize)
            a = px[np.sort(np.random.default_rng(seed).choice(px.shape[0], n, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------- post-pass leg
def post_leg(W, H, tris):
    """Informational, run in its OWN process by the default single-GPU bench (crash isolation: these kernels had no GPU time before the
    round-end run): deferred combine -> TAA -> tone map and the ground-truth path tracer at the bench resolution, CUDA-event timed.
    Prints one JSON dict.  Algorithmic bytes per pixel (DESIGN.md section 5): TAA 36, tone map 12."""
    import torch
    import pyhr
    torch.cuda.set_device(0)
    ctx = pyhr.Context(0)
    ctx.set_bluenoise(*pyhr.blue_noise())
    sc = pyhr.SynthScene(pyhr.SCENE_ARCADE, tris)
    ctx.current_scene_handle = ctx.build_scene(sc)
    ctx.gbuffer_create(W, H)
    light = pyhr.default_light(rot_x_deg=LIGHT_ROT_X)
    stream = torch.cuda.current_stream().cuda_stream
    f = pyhr.make_frame(CAM_POS, CAM_TGT, W, H, light=light)
    f = pyhr.make_frame(CAM_POS, CAM_TGT, W, H, prev=f, num_frames=1, light=light)
    ctx.gbuffer_render(0, f, 0, 0, stream)
    ctx.gbuffer_render(1, f, 0, 0, stream)
    de, taa, tm, pt = pyhr.DeferredPass(ctx, W, H), pyhr.TAAPass(ctx, W, H), pyhr.TonemapPass(ctx, W, H), pyhr.PathTracerPass(ctx, W, H)
    for k in range(3):
        de.params.env_color[k] = pt.params.sky_color[k] = SKY[k]
    j = pyhr.taa_jitter(1, W, H)
    f.ubo.current_prev_jitter[0], f.ubo.current_prev_jitter[1] = float(j[0]), float(j[1])

    def timed(fn, n, warm=3):
        for _ in range(warm):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    peak, peak_src = read_peaks()
    px = float(W * H)
    out = {"width": W, "height": H, "triangles": tris, "peak_source": peak_src}
    out["deferred_ms"] = timed(lambda: de.render(f, None, None, None, None, stream), 20)
    taa.params.reset_every_frame = 0
    t = timed(lambda: taa.render(f, de, stream), 20)
    out["taa"] = {"ms": t, "algorithmic_bytes": 36.0 * px, "achieved_gbs": 36.0 * px / 1e9 / (t / 1e3), "frac": 36.0 * px / 1e9 / (t / 1e3) / peak}
    taa.params.reset_every_frame = 1
    out["taa_with_reset_blit_ms"] = timed(lambda: taa.render(f, de, stream), 20)
    t = timed(lambda: tm.render(taa, stream), 20)
    out["tonemap"] = {"ms": t, "algorithmic_bytes": 12.0 * px, "achieved_gbs": 12.0 * px / 1e9 / (t / 1e3), "frac": 12.0 * px / 1e9 / (t / 1e3) / peak}
    pt.stats(stream)
    t = timed(lambda: pt.render(f, stream), 8, warm=2)
    st = pt.stats(stream)
    rays = (st.rays_primary + st.rays_secondary) / max(1, st.renders)
    out["path_tracer"] = {"ms_per_sample": t, "rays_per_sample": rays, "mrays_per_s": rays / 1e6 / (t / 1e3)}
    ldr = tm.download(100)
    out["tonemapped_mean"] = float(ldr[..., :3].mean())
    out["launches"] = ctx.launch_count()
    try:
        # material textures (hr_scene_set_textures): cost of the TEX instantiations of the G-buffer producer and of the reflections ray trace
        # against the untextured kernels, same frame; a 1024 x 1024 sRGB albedo, a packed roughness / metallic image and a normal map on every material
        rng = np.random.default_rng(7)
        yy, xx = np.mgrid[0:1024, 0:1024]
        albedo = np.stack([np.where((xx // 64 + yy // 64) % 2, 220, 60), (xx // 4) % 256, (yy // 4) % 256, np.full_like(xx, 255)], -1).astype(np.uint8)
        orm = rng.integers(0, 256, (512, 512, 4), dtype=np.uint8)
        bump = np.stack([128 + (40 * np.sin(xx[:256, :256] * 0.2)).astype(int), 128 + (40 * np.cos(yy[:256, :256] * 0.2)).astype(int),
                         np.full((256, 256), 235), np.full((256, 256), 255)], -1).astype(np.uint8)
        rf = pyhr.ReflectionsPass(ctx, W, H, 0)
        src = refl_params(CONFIGS[3])
        for name, _ in src._fields_:
            if name != "sky_color":
                setattr(rf.params, name, getattr(src, name))
        for k in range(3):
            rf.params.sky_color[k] = SKY[k]
        rf.params.denoise = 0

        def frame_cost():
            ctx.set_profiling(True)
            g_ms = timed(lambda: ctx.gbuffer_render(f.ping_pong, f, 0, 0, stream), 10)
            rf.stage_times()
            for _ in range(6):
                rf.render(f, None, stream)
            torch.cuda.synchronize()
            st = dict(rf.stage_times())
            ctx.set_profiling(False)
            return g_ms, st.get("Ray Trace")

        plain = frame_cost()
        scene_ptr = ctx.current_scene_handle
        ctx.set_textures(scene_ptr, [(albedo, True), (orm, False), (bump, False)],
                         [dict(albedo=0, roughness=1, roughness_channel=1, metallic=1, metallic_channel=2, normal=2)] * sc.n_materials)
        textured = frame_cost()
        out["textured"] = {"gbuffer_ms": {"constants": plain[0], "textures": textured[0]}, "reflections_ray_trace_ms": {"constants": plain[1], "textures": textured[1]},
                           "textures": "1024x1024 sRGB albedo + 512x512 roughness/metallic + 256x256 normal map on every material"}
        rf.destroy()
    except Exception as e:  # informational: keep what was measured above
        out["textured"] = {"error": f"{type(e).__name__}: {e}"}
    try:
        for p in (de, taa, tm, pt):
            p.destroy()
        ctx.close()
    except Exception:
        pass
    print(json.dumps(out))


def run_post_leg(W, H, tris):
    import subprocess
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--post-leg", str(W), str(H), str(tris)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                           timeout=240, env={**os.environ, "CUDA_VISIBLE_DEVICES": os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]})
        if r.returncode != 0:
            return {"error": f"exit code {r.returncode}: {r.stderr.strip()[-400:]}"}
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:  # informational leg: never takes the bench line down
        return {"error": f"{type(e).__name__}: {e}"}


def main():
    if len(sys.argv) == 5 and sys.argv[1] == "--post-leg":
        return post_leg(int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]))
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the pan / dense-K5 / host-G-buffer legs (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write every pass's final output of the last step as DIR/<pass>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    cfg = CONFIGS[args.config]
    W, H = cfg["W"], cfg["H"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    metric = f"denoised frames/s @{'4K' if W == 3840 else '%dx%d' % (W, H)} ({'+'.join(cfg['passes'])}, {cfg.get('spp', 1)} spp" + (", full SVGF)" if cfg.get("denoise", True) else ", no denoise)")
    config = {"workload": f"config {args.config}: {cfg['name']}; static camera steady state", "baseline_config": args.config, "width": W, "height": H,
              "triangles": cfg["tris"], "passes": cfg["passes"], "spp": cfg.get("spp", 1), "parallelism": f"row-band x{world}", "l2_policy": "inputs_larger_than_l2"}

    if args.impl == "reference":
        # The reference has no CPU implementation of this path (SURVEY.md fact 4) and cannot be built here (Vulkan RT + GLSL):
        # this arm times the CPU oracle, a port, with every host thread on a bounded sample of the same workload.
        if rank != 0:
            return
        cb = oracle_fps(cfg, frames=max(1, min(args.steps, 5)))
        line = {"metric": metric, "value": cb["value"], "unit": "frames/s", "n_gpus": args.gpus, "steps": max(1, min(args.steps, 5)), "warmup": 1,
                "ms_per_step": 1000.0 / cb["value"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (fp16 storage)", "data": "synthetic",
                "config": config, "impl": "reference", "cpu_baseline": cb,
                "note": "cpu oracle (port), measured on a reduced-area sample and extrapolated; NOT the upstream implementation (it has no CPU path)",
                "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import pyhr

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- scene, context ------------------------------------------------------------------------------------------------------
    single_tri = cfg.get("scene") == "single_triangle"
    if single_tri:
        light = pyhr.default_light()
        sc, gsc = pyhr.SynthScene(pyhr.SCENE_SINGLE_TRIANGLE), pyhr.SynthScene(pyhr.SCENE_GROUND_PLANE)
        cam, tgt = (0.0, 8.0, 20.0), (0.0, 0.0, 0.0)
    else:
        light = pyhr.default_light(rot_x_deg=LIGHT_ROT_X)
        sc = gsc = pyhr.SynthScene(pyhr.SCENE_ARCADE, cfg["tris"])
        cam, tgt = CAM_POS, CAM_TGT
    ctx = pyhr.Context(local_rank)
    for env, key in (("HR_ATROUS_IMPL", 1), ("HR_TRACE_IMPL", 2), ("HR_BVH_QUALITY", 3), ("HR_FORCE_SHARED_RT", 4), ("HR_ATROUS_ROWS", 5), ("HR_REFL_ATROUS_IMPL", 6), ("HR_REFL_TRACE_IMPL", 7), ("HR_REFL_ATROUS_MINB", 8), ("HR_SHADOW_PACKET", 9), ("HR_REFL_TRACE_MINB", 10), ("HR_GATHER_IMPL", 11), ("HR_FORCE_PEER_TEMPORAL", 12)):
        if os.environ.get(env):
            ctx.lib.hr_debug_set(key, int(os.environ[env]))
    ctx.set_bluenoise(*pyhr.blue_noise())
    if world > 1:
        uid = [pyhr.shard_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.shard_init(rank, world, uid[0])
    t_b = time.perf_counter()
    scene_h = ctx.build_scene(sc)
    torch.cuda.synchronize()
    build_ms = (time.perf_counter() - t_b) * 1e3
    ctx.gbuffer_create(W, H)
    rig = Rig(pyhr, ctx, cfg, W, H)
    stream = torch.cuda.current_stream().cuda_stream
    state = {"f": None, "n": 0, "x": 0.0}

    def next_frame(dx=0.0):
        state["x"] += dx
        pos = (cam[0] + state["x"], cam[1], cam[2])
        state["f"] = pyhr.make_frame(pos, tgt, W, H, prev=state["f"], num_frames=state["n"], light=light)
        state["n"] += 1
        return state["f"]

    # ---- G-buffer of the static view, resident in both slots -----------------------------------------------------------------------
    g_host = None
    f0 = next_frame()
    f1 = next_frame()
    if single_tri:
        g_host = pyhr.write_gbuffer(gsc, f1, W, H, pinned=True)
        ctx.gbuffer_upload(0, g_host, stream)
        ctx.gbuffer_upload(1, g_host, stream)
    else:
        ctx.gbuffer_render(0, f1, 0, 0, stream)
        ctx.gbuffer_render(1, f1, 0, 0, stream)

    def step_resident():
        rig.render(next_frame(), stream)

    def gather(on):
        if world > 1:
            ctx.shard_set_gather(on)

    # history warm-up to steady state (history length saturates at 32)
    gather(True)
    n_warm = max(args.warmup, 3) + 32
    for _ in range(n_warm):
        step_resident()
    torch.cuda.synchronize()

    def timed(fn, steps, profile=False, sample=False, finish=None):
        if profile:
            rig.stage_times()
            ctx.set_profiling(True)
        sampler = ClockSampler(local_rank) if sample else None
        l0 = ctx.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        if sampler:
            sampler.start()
        e0.record()
        for _ in range(steps):
            fn()
        if finish:
            finish()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        out = {"ms": ms, "launches": ctx.launch_count() - l0, "clocks": sampler.result() if sampler else None}
        if profile:
            out["stages"] = rig.stage_times()
            ctx.set_profiling(False)
        return out

    # ---- value: resident G-buffer; N > 1: final outputs gathered to every rank inside the timed region -----------------------------
    rig.stats(stream)  # reset the ray counters
    r_val = timed(step_resident, args.steps, profile=True, sample=True)
    st_val = rig.stats(stream)
    if args.dump_outputs and rank == 0:  # the final outputs are gathered: rank 0 holds whole frames
        dump_outputs(args.dump_outputs, {name: p.download(100, stream) for name, p in rig.passes.items()})
    r_dist = None
    if world > 1:
        gather(False)
        for _ in range(3):
            step_resident()
        r_dist = timed(step_resident, args.steps, profile=True)
        gather(True)

    # ---- outputs / staging for the host legs -----------------------------------------------------------------------------------------
    outs = []
    for name, p in rig.passes.items():
        img = p.output(100)
        b0, b1 = pyhr.shard_rows(H, rank, world)  # this rank's band, scaled to the image's own height (ray masks: H / 4 rows)
        b0, b1 = b0 * img.height // H, (img.height if b1 >= H else b1 * img.height // H)
        nbytes = (b1 - b0) * img.width * texel_bytes(img)
        dev = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        host = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        outs.append((p, b0, b1, dev, host, nbytes))
    d2h_bytes = sum(o[5] for o in outs)
    s_copy = torch.cuda.Stream()
    ev_staged, ev_copied = torch.cuda.Event(), torch.cuda.Event()
    ev_copied.record(torch.cuda.current_stream())
    cur = torch.cuda.current_stream()

    def read_back():
        # stage the final outputs on the device behind the frame's kernels (a few tens of microseconds), then let the PCIe copy
        # run on its own stream while the next frame renders; the next staging waits for the previous copy
        cur.wait_event(ev_copied)
        for p, b0, b1, dev, host, nb in outs:
            p.lib.hr_pass_download_rows_async(p.h, 100, b0, b1, C.c_void_p(dev.data_ptr()), C.c_size_t(nb), C.c_void_p(stream))
        ev_staged.record(cur)
        s_copy.wait_event(ev_staged)
        with torch.cuda.stream(s_copy):
            for p, b0, b1, dev, host, nb in outs:
                host.copy_(dev, non_blocking=True)
            ev_copied.record(s_copy)

    pipelined = world == 1 and not single_tri  # the next frame's G-buffer ray cast runs on the library's side stream under this frame's passes

    def step_e2e():
        if pipelined:
            f = state["staged"]
            ctx.gbuffer_commit_staged(f.ping_pong, stream)
            state["staged"] = next_frame()
            ctx.gbuffer_stage_render(state["staged"])
        else:
            f = next_frame()
            if single_tri:
                ctx.gbuffer_upload(f.ping_pong, g_host, stream)
            elif cfg["passes"] == ["reflections"] and cfg.get("refl_scale", 1) == 0:
                ctx.gbuffer_render_sharded(f.ping_pong, f, 64, stream)  # only the rows this rank's stages read (band +- 64, its ray-trace chunks)
            else:
                ctx.gbuffer_render(f.ping_pong, f, 0, 0, stream)
        rig.render(f, stream)
        read_back()

    if pipelined:
        state["staged"] = next_frame()
        ctx.gbuffer_stage_render(state["staged"])

    gather(False)  # e2e: every rank reads its own band back to its host
    for _ in range(3):
        step_e2e()
    r_e2e = timed(step_e2e, args.steps, finish=lambda: cur.wait_event(ev_copied))  # the last frame's PCIe copy is inside the timed region
    if pipelined:  # retire the frame staged by the last step (never rendered: it pays back the one staged before the clock started)
        ctx.gbuffer_commit_staged(state["staged"].ping_pong, stream)
        state["f"] = state["staged"]
        torch.cuda.synchronize()
    h2d_bytes = int(g_host.nbytes()) if single_tri else C.sizeof(pyhr.hr_frame)

    extras = {}
    if not args.no_extras and not single_tri:
        # ---- pan: 40 frames of lateral motion, G-buffer produced on the device every frame --------------------------------------------
        sharded_gbuf = world > 1 and cfg["passes"] == ["reflections"] and cfg.get("refl_scale", 1) == 0

        def step_pan():
            f = next_frame(PAN_STEP)
            if sharded_gbuf:  # as in the e2e leg: only the rows this rank's stages read (the pan is lateral: reprojection stays within the 64-row halo)
                ctx.gbuffer_render_sharded(f.ping_pong, f, 64, stream)
            else:
                ctx.gbuffer_render(f.ping_pong, f, 0, 0, stream)
            rig.render(f, stream)

        gather(True)
        for _ in range(8):
            step_pan()
        ge0, ge1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r_pan = timed(step_pan, 40, profile=True)
        # the G-buffer producer alone
        barrier()
        ge0.record()
        for _ in range(10):
            if sharded_gbuf:
                ctx.gbuffer_render_sharded(state["f"].ping_pong, state["f"], 64, stream)
            else:
                ctx.gbuffer_render(state["f"].ping_pong, state["f"], 0, 0, stream)
        ge1.record()
        torch.cuda.synchronize()
        extras["pan"] = {"frames": 40, "step_world_units": PAN_STEP, "ms": r_pan["ms"], "gbuffer_ms_per_frame": ge0.elapsed_time(ge1) / 10.0, "stages": r_pan["stages"]}
        # ---- host G-buffer mode of the e2e leg (upload GB2 + GB3 + depth every frame; GB1 is not read by these passes) -----------------
        if world == 1:
            gh = pyhr.GBufferHost(W, H, pinned=True)
            for which, arr in ((2, gh.gb2), (3, gh.gb3), (0, gh.depth)):
                arr[...] = ctx.gbuffer_download(state["f"].ping_pong, 0, which, W, H)
            gh_desc = pyhr.hr_gbuffer_desc(W, H, None, gh.gb2.ctypes.data_as(C.c_void_p), gh.gb3.ctypes.data_as(C.c_void_p), gh.depth.ctypes.data_as(C.c_void_p))

            def step_e2e_host():
                f = next_frame()
                ctx.check(ctx.lib.hr_gbuffer_commit_staged(ctx.h, f.ping_pong, C.c_void_p(stream)), "hr_gbuffer_commit_staged")
                ctx.check(ctx.lib.hr_gbuffer_stage_upload(ctx.h, C.byref(gh_desc)), "hr_gbuffer_stage_upload")
                rig.render(f, stream)
                read_back()

            ctx.check(ctx.lib.hr_gbuffer_stage_upload(ctx.h, C.byref(gh_desc)), "hr_gbuffer_stage_upload")
            for _ in range(3):
                step_e2e_host()
            r_host = timed(step_e2e_host, min(args.steps, 20), finish=lambda: cur.wait_event(ev_copied))
            extras["e2e_host_gbuffer"] = {"value": min(args.steps, 20) / (r_host["ms"] / 1e3), "h2d_bytes_per_step": W * H * 20}
            ctx.check(ctx.lib.hr_gbuffer_commit_staged(ctx.h, state["f"].ping_pong, C.c_void_p(stream)), "hr_gbuffer_commit_staged")
            torch.cuda.synchronize()

    # ---- N > 1: the gathered frame equals the single-GPU frame (device checksums of the final outputs) -----------------------------------
    parity = None
    if world > 1:
        gather(True)
        rig.reset()
        state.update(f=None, n=0, x=0.0)
        fr = [next_frame() for _ in range(6)]
        if not single_tri:
            ctx.gbuffer_render(0, fr[1], 0, 0, stream)
            ctx.gbuffer_render(1, fr[1], 0, 0, stream)
        for f in fr[2:]:
            rig.render(f, stream)
        torch.cuda.synchronize()
        sums = {k: p.checksum(100, 0, 0, stream) for k, p in rig.passes.items()}
        mine = torch.tensor([v & 0x7FFFFFFFFFFFFFFF for v in sums.values()], dtype=torch.int64, device="cuda")
        allv = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        ranks_agree = all(bool((a == allv[0]).all()) for a in allv)
        ref_ok = None
        if rank == 0:
            c1 = pyhr.Context(local_rank)
            c1.set_bluenoise(*pyhr.blue_noise())
            s1 = c1.build_scene(sc)
            c1.gbuffer_create(W, H)
            rig1 = Rig(pyhr, c1, cfg, W, H)
            if not single_tri:
                c1.gbuffer_render(0, fr[1], 0, 0, stream)
                c1.gbuffer_render(1, fr[1], 0, 0, stream)
            for f in fr[2:]:
                rig1.render(f, stream)
            torch.cuda.synchronize()
            sums1 = {k: p.checksum(100, 0, 0, stream) for k, p in rig1.passes.items()}
            ref_ok = sums1 == sums
            rig1.destroy()
            c1.lib.hr_scene_destroy(s1)
            c1.close()
        parity = {"frames": 4, "ranks_agree": ranks_agree, "equals_single_gpu": ref_ok}

    # ---- dense-penumbra K5 (single GPU line only): shadows pass alone at this resolution on a view with >= 95 % denoise tiles -------------
    k5_dense = None
    if not args.no_extras and world == 1 and not single_tri:
        rig.destroy()
        rig = None
        ctx.lib.hr_scene_destroy(scene_h)
        sc2 = pyhr.SynthScene(pyhr.SCENE_SHADOWS_TEST)
        scene_h = ctx.build_scene(sc2)
        shp = pyhr.Pass(ctx, "shadows", W, H, 0)
        fa = pyhr.make_frame(DENSE_CAM[0], DENSE_CAM[1], W, H, light=light)
        fb = pyhr.make_frame(DENSE_CAM[0], DENSE_CAM[1], W, H, prev=fa, num_frames=1, light=light)
        ctx.gbuffer_render(0, fb, 0, 0, stream)
        ctx.gbuffer_render(1, fb, 0, 0, stream)
        fd = fb
        for i in range(40):
            fd = pyhr.make_frame(DENSE_CAM[0], DENSE_CAM[1], W, H, prev=fd, num_frames=2 + i, light=light)
            shp.render(fd, stream)
        torch.cuda.synchronize()
        ctx.set_profiling(True)
        shp.stage_times()
        for i in range(20):
            fd = pyhr.make_frame(DENSE_CAM[0], DENSE_CAM[1], W, H, prev=fd, num_frames=42 + i, light=light)
            shp.render(fd, stream)
        torch.cuda.synchronize()
        sts = dict(shp.stage_times())
        ctx.set_profiling(False)
        s5 = shp.stats(stream)
        at = [v for k, v in sts.items() if k.startswith("A-Trous")]
        on, tot = s5.tiles_denoise, max(1, s5.tiles_total)
        b_on, b_off = ATROUS_BYTES["shadows"]
        proc = 64.0 * (on * b_on + (tot - on) * b_off)
        peak, _ = read_peaks()
        k5_dense = {"workload": f"{W}x{H} shadows pass on the shadows-test scene seen from above", "tiles_on_denoise_list_frac": on / tot,
                    "avg_launch_ms": float(np.mean(at)), "per_iteration_ms": at, "processed_bytes_per_launch": proc,
                    "achieved": proc / 1e9 / (float(np.mean(at)) / 1e3), "frac": proc / 1e9 / (float(np.mean(at)) / 1e3) / peak, "stages_ms": sts}
        shp.destroy()

    # ---- reduce over ranks ----------------------------------------------------------------------------------------------------------------
    vals = [r_val["ms"], r_e2e["ms"], r_dist["ms"] if r_dist else 0.0, extras.get("pan", {}).get("ms", 0.0)]
    t = torch.tensor(vals, dtype=torch.float64, device="cuda")
    stage_sum = {k: sum(v.values()) for k, v in r_val["stages"].items()}
    busy = torch.tensor([sum(stage_sum.values()), sum(v.get("Ray Trace", 0.0) for v in r_val["stages"].values()),
                         sum(sum(x for n, x in v.items() if "Wait" in n) for v in r_val["stages"].values())], dtype=torch.float64, device="cuda")
    busy_all = [busy.clone() for _ in range(world)]
    rank_stages = None
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_gather(busy_all, busy)
        # per-rank stage times of the gathered and of the distributed leg (which rank waits for whom)
        rank_stages = [None] * world
        dist.all_gather_object(rank_stages, {"gathered": r_val["stages"], "distributed": r_dist["stages"] if r_dist else None})
    ms_val, ms_e2e, ms_dist, ms_pan = [float(x) for x in t]

    if rank == 0:
        peak, peak_src = read_peaks()
        key = "reflections" if "reflections" in cfg["passes"] else "shadows"
        kname = "k_refl_atrous (reflections a-trous, K16)" if key == "reflections" else "k_atrous_v3 (shadows a-trous, K5)"
        st = r_val["stages"].get(key, {})
        at = [v for k, v in st.items() if k.startswith("A-Trous")]
        roof = None
        if at:
            s = st_val[key]
            at_ms = float(np.mean(at))
            b_on, b_off = ATROUS_BYTES[key]
            on, tot = s.tiles_denoise, max(1, s.tiles_total)
            proc = 64.0 * (on * b_on + (tot - on) * b_off)
            contract = b_on * s.pixels_total
            tr = read_traffic(key)
            roof = {"kernel": kname, "bound": "hbm", "achieved": proc / 1e9 / (at_ms / 1e3), "peak": peak, "unit": "GB/s", "frac": proc / 1e9 / (at_ms / 1e3) / peak,
                    "frac_contract": contract / 1e9 / (at_ms / 1e3) / peak, "avg_launch_ms": at_ms, "per_iteration_ms": at,
                    "algorithmic_bytes_per_launch": proc, "contract_bytes_per_launch": contract, "bytes_per_px": {"denoise_tile": b_on, "other_tile": b_off},
                    "tiles_total": int(tot), "tiles_on_denoise_list": int(on), "peak_source": peak_src,
                    "traffic": tr[0] if (tr and world == 1) else None, "traffic_source": (f"{tr[1]} ({tr[2]})" if tr else None)}
        rays = {k: {"primary_per_frame": s.rays_primary / max(1, s.renders), "secondary_per_frame": s.rays_secondary / max(1, s.renders),
                    "trace_kernel_ms": r_val["stages"].get(k, {}).get("Ray Trace"),
                    "mrays_per_s": ((s.rays_primary + s.rays_secondary) / max(1, s.renders) / 1e6) / (r_val["stages"][k]["Ray Trace"] / 1e3)
                    if r_val["stages"].get(k, {}).get("Ray Trace") else None} for k, s in st_val.items()}
        fps = args.steps / (ms_val / 1e3)
        line = {
            "metric": metric, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": n_warm, "ms_per_step": ms_val / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (fp16 storage)", "data": "synthetic", "config": config,
            "clocks": r_val["clocks"], "gpu_launches": int(r_val["launches"]),
            "e2e": {"value": args.steps / (ms_e2e / 1e3), "unit": "frames/s", "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes),
                    "mode": ("host G-buffer upload (the analytic plane is not in the BVH)" if single_tri else
                             "host hr_frame -> G-buffer ray cast on the device (pipelined one frame ahead on a side stream when N = 1) -> passes -> outputs staged and copied to pinned host memory on a copy stream"),
                    "host_gbuffer_value": extras.get("e2e_host_gbuffer", {}).get("value"), "host_gbuffer_h2d_bytes_per_step": extras.get("e2e_host_gbuffer", {}).get("h2d_bytes_per_step")},
            "roofline": roof, "stages_ms": r_val["stages"], "mrays_per_s": rays, "scene_build_ms": build_ms,
            "rank_busy_ms": [{"stage_sum": round(float(b[0]), 4), "ray_trace": round(float(b[1]), 4), "waits": round(float(b[2]), 4)} for b in busy_all],
        }
        if world > 1:
            line["value_gathered"] = fps
            line["value_distributed"] = args.steps / (ms_dist / 1e3)
            line["rank_stages_ms"] = [{leg: ({pn: {k: round(v, 4) for k, v in st.items()} for pn, st in d.items()} if d else None) for leg, d in rs.items()}
                                      for rs in rank_stages]
            line["parity_crc_ok"] = bool(parity and parity["ranks_agree"] and parity["equals_single_gpu"])
            line["parity"] = parity
        if "pan" in extras:
            line["pan"] = {"value": 40 / (ms_pan / 1e3), "unit": "frames/s", "frames": 40, "world_units_per_frame": PAN_STEP,
                           "gbuffer_ms_per_frame": extras["pan"]["gbuffer_ms_per_frame"], "stages_ms": extras["pan"]["stages"],
                           "note": "includes the G-buffer ray cast every frame (N > 1: hr_gbuffer_render_sharded, this rank's rows only)"}
        if k5_dense:
            line["k5_dense"] = k5_dense
        if not args.no_extras and world == 1 and not single_tri:
            # deferred -> TAA -> tone map and the ground-truth path tracer (SURVEY.md section 8 f2 / f4), timed in a separate process
            line["post_passes"] = run_post_leg(W, H, cfg["tris"])
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = oracle_fps(cfg)
        print(json.dumps(line))
    if rig:
        rig.destroy()
    ctx.lib.hr_scene_destroy(scene_h)
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
