#!/usr/bin/env python
"""bench.py — Mrays/s of the path-tracing hot path on B200 (BASELINE.json metric).

Default workload ("4k"): the 4K offline screenshot BASELINE.json's north star names for the multi-GPU target —
BASELINE config 5 at a stated QUARTER of its samples: the config-2 scene (Cornell box + 100 352-triangle textured
mesh) at 3840x2160, 1024 spp = 16 frames x 64 spp (`screenshot()`'s unit, rayTracing.cpp:68-72,184-242), max depth 20,
Philox RNG.  The job is FIXED whatever the GPU count (strong scaling): N ranks share the 16 frames (frame f on rank
f % N, the same frameIndex a single GPU uses), the 8-bit frame sums are reduced to rank 0 over NCCL inside the
library, rank 0 finalizes.  A step = one whole screenshot: raygen -> [extend -> shade] x depth -> accumulate ->
resolve per frame -> (reduce) -> finalize.

`value` times the step with the scene resident in HBM (rt_screenshot_device); `e2e` times the whole job from HOST
buffers through the C-ABI (triangle / material / texture upload, BVH build, rt_screenshot with the RGB8 image copied
back).  At N = 1 the line also carries `config2` (the 1080p / 256 spp case of BASELINE config 2, round 1's headline)
and `config4` (10 M triangles at 4K, 2 of its 16 frames: the HBM-bound case), each with its own roofline block.

`roofline` is for the dominant kernel (k_extend) against the ceiling that BINDS: the largest of
t_hbm (path records streamed + BVH bytes if the BVH does not fit L2, at the measured copy peak),
t_gather (BVH node + triangle bytes at the measured random-gather bandwidth for a table of the BVH's size:
tools/microbench.cu, run inside this process just before the timed region) and
t_fp32 (box + triangle test flops at the measured non-FMA FP32 issue rate) — SURVEY.md §8d's max(...).

--impl reference: the reference's own compute shader compiled for the CPU (oracle/_ref/libref_shader_libm.so) on all
host threads, on a bounded sample of the same workload; the oracle port if that library is absent.
"""
from __future__ import annotations

import argparse
import ctypes
import importlib
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
for p in (REPO, os.path.join(REPO, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

# name -> image, frames of 64 spp, depth, scene.  "4k" is the bench line; the others are the BASELINE configs
# (`--workload` measures them for the record, config2 / config4 also ride along in the default line at N = 1).
WORKLOADS = {
    "4k": dict(width=3840, height=2160, frames=16, max_bounce=20, scene="sphere_cornell",
               text="BASELINE config 5 at a quarter of its samples: config-2 scene (addCornellBox 0.17/0.3, light 15.0 + "
                    "synthetic textured displaced sphere, 100 352 + 16 triangles), 3840x2160, 1024 spp = 16 frames x 64 spp "
                    "in total (fixed for every GPU count), max depth 20, environmentalLight 0"),
    "config1": dict(width=512, height=512, frames=1, max_bounce=8, scene="classic",
                    text="BASELINE config 1: classic Cornell box, 38 triangles, 512x512, 64 spp, depth 8"),
    "config2": dict(width=1920, height=1080, frames=4, max_bounce=20, scene="sphere_cornell",
                    text="BASELINE config 2: Cornell box + synthetic textured displaced sphere (100 352 + 16 triangles), "
                         "1920x1080, 256 spp = 4 frames x 64 spp, depth 20"),
    "config3": dict(width=1920, height=1080, frames=8, max_bounce=16, scene="sphere_mirror",
                    text="BASELINE config 3: full-mirror box + the same mesh, 1920x1080, 512 spp = 8 frames x 64 spp, depth 16"),
    "config4": dict(width=3840, height=2160, frames=16, max_bounce=8, scene="big_sphere",
                    text="BASELINE config 4: 9 999 392-triangle displaced sphere in the classic Cornell room, 3840x2160, "
                         "1024 spp = 16 frames x 64 spp, depth 8"),
    "config2_robot": dict(width=1920, height=1080, frames=4, max_bounce=20, scene="robot",
                          text="BASELINE config 2(i): Data/robot (25 599 triangles, 3 textures) in addCornellBox, 1920x1080, "
                               "256 spp, depth 20 (needs tools/make_assets.sh)"),
}
SPP_PER_FRAME = 64
N_QUADS, TEX_SIZE = 224, 1024
CPU_SAMPLE = dict(crop_frac=4, frames=1, paths=518400)  # centred crop of 1/4 x 1/4 of the image, ~0.5 M camera paths
# --dump-outputs: at most this many pixels of the screenshot (2 Mi x (3 x f32 + f64 index) = 40 MiB), picked by a fixed seed
DUMP_PIXELS, DUMP_SEED = 1 << 21, 0


def build_scene(rt, name):
    wl = WORKLOADS[name]
    W, H = wl["width"], wl["height"]
    kind = wl["scene"]
    if kind == "classic":
        scene = rt.scene_classic_cornell()
        cam = rt.make_camera(W, H, (0.0, 0.0, 15.5))
    elif kind == "sphere_mirror":
        scene = rt.scene_textured_sphere(n_quads=N_QUADS, container="mirror", tex_size=TEX_SIZE)
        cam = rt.camera_for_box(scene, W, H)
    elif kind == "robot":
        scene = rt.scene_from_rtsc(os.path.join(REPO, "assets", "_gen", "robot.rtsc"), container="cornell")
        cam = rt.camera_for_box(scene, W, H)
    elif kind == "big_sphere":
        scene = rt.scene_big_sphere(n_quads=2236)
        cam = rt.make_camera(W, H, (0.0, 0.0, 15.5))
    else:
        scene = rt.scene_textured_sphere(n_quads=N_QUADS, container="cornell", tex_size=TEX_SIZE)
        cam = rt.camera_for_box(scene, W, H)
    u = rt.screenshot_uniforms(scene, cam, spp=SPP_PER_FRAME, max_bounce=wl["max_bounce"], env_light=False)
    return scene, cam, u


def workload_config(name, frames_total, n_gpus, split):
    wl = WORKLOADS[name]
    return {
        "workload": wl["text"],
        "name": name,
        "rng": "philox4x32-10 keyed (pixel, frame, sample, bounce, draw)",
        "frames_total": int(frames_total),
        "split": "frame-slice (frame f on rank f % N) + ncclReduce of the 8-bit frame sums to rank 0" if split == "frames"
                 else "image-tile (bands of 8 rows dealt round-robin) + gather of each rank's rows to rank 0",
        "cache": "the path state of one wavefront batch (up to 512 Mi paths x 128 B = 64 GiB) is far larger than the "
                 "126 MB L2 and is rewritten every bounce: inputs larger than L2, no explicit flush",
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", os.environ.get("RT_BENCH_CLOCK_MS", "100")],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); smax.append(float(r[1])); power.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def git_head():
    try:
        return subprocess.check_output(["git", "-C", REPO, "rev-parse", "--short=12", "HEAD"], text=True,
                                       stderr=subprocess.DEVNULL).strip()
    except Exception:
        return None


def microbench(extend_blocks_per_sm):
    """The ceilings, measured now on this GPU (tools/microbench.cu): random-gather bandwidth for 32 B / 64 B records
    out of an 8 MB (L2-resident) and a 1 GB (HBM-resident) table at k_extend's residency, the issue rate of the
    instruction classes the node step is made of, and a plain copy."""
    path = os.path.join(REPO, "tools", "libmicrobench.so")
    if not os.path.exists(path):
        return {"error": "tools/libmicrobench.so missing (make -C tools)"}
    L = ctypes.CDLL(path)
    L.mb_gather_gbs.restype = ctypes.c_double
    L.mb_gather_gbs.argtypes = [ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    L.mb_issue_tops.restype = ctypes.c_double
    L.mb_issue_tops.argtypes = [ctypes.c_int, ctypes.c_int]
    L.mb_stream_gbs.restype = ctypes.c_double
    L.mb_stream_gbs.argtypes = [ctypes.c_size_t]
    bps = int(extend_blocks_per_sm)
    out = {"when": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()), "git": git_head(),
           "resident_threads_per_sm": bps * 128, "gather_gbs": {}, "issue_tops": {}}
    for table, tname in ((8 << 20, "8MB"), (1 << 30, "1GB")):
        for rec in (32, 64):
            for dep in (0, 1):
                key = f"{tname}_{rec}B_{'dependent' if dep else 'independent'}"
                out["gather_gbs"][key] = L.mb_gather_gbs(table, rec, dep, bps, 256 if dep == 0 else 512)
    for kind, kname in enumerate(("fadd_fmul", "ffma", "fmnmx", "i2f_u16", "slab_mix")):
        out["issue_tops"][kname] = L.mb_issue_tops(kind, 4096)
    out["stream_copy_gbs"] = L.mb_stream_gbs(1 << 30)
    return out


def dump_outputs(out_dir, shot):
    """What the timed path hands its caller, the RGB8 screenshot (H, W, 3), as .npy files that two builds can be
    compared on: screenshot.npy holds the RGB values (float32, one row per pixel) of up to DUMP_PIXELS pixels drawn
    without replacement by a fixed seed, screenshot_pixel_index.npy their row-major pixel indices (float64, ascending).
    An image of at most DUMP_PIXELS pixels is written whole."""
    os.makedirs(out_dir, exist_ok=True)
    rgb = shot.reshape(-1, 3)
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(rgb.shape[0], size=min(rgb.shape[0], DUMP_PIXELS), replace=False))
    np.save(os.path.join(out_dir, "screenshot.npy"), rgb[idx].astype(np.float32))
    np.save(os.path.join(out_dir, "screenshot_pixel_index.npy"), idx.astype(np.float64))


def pinned_copy(torch, a: np.ndarray):
    """The same bytes in page-locked host memory (numpy view of a pinned torch tensor)."""
    t = torch.empty(max(a.nbytes, 1), dtype=torch.uint8, pin_memory=True)
    v = t.numpy()[: a.nbytes]
    v[:] = np.frombuffer(a.tobytes(), dtype=np.uint8)
    return v.view(a.dtype).reshape(a.shape), t  # keep `t` alive as long as the view is used


# ------------------------------------------------------------------------------------------------ CPU arm
_CPU_ARM = {}


def cpu_region(W, H):
    f = CPU_SAMPLE["crop_frac"]
    cw, ch = W // f, H // f
    x0, y0 = (W - cw) // 2, (H - ch) // 2
    spp = max(1, CPU_SAMPLE["paths"] // (cw * ch))
    return (x0, y0, x0 + cw, y0 + ch), spp


def cpu_arm(rt, name):
    """The CPU implementation that gets timed, prepared once: the reference's OWN compute shader source
    (oracle/_ref/libref_shader_libm.so: compute.glsl rewritten syntactically by oracle/glsl2cpp.py, compiled with
    g++ -O2 against the reference's glm, libm elementary functions; built where /root/reference exists and shipped
    prebuilt) over the reference's BVH — `kind: "reference"`.  If that library is missing the oracle port is
    timed instead — `kind: "port"`.  Either way the segment count comes from the oracle on the identical frame
    (RT_RNG_REF_PCG: the oracle's frame is bit-identical to the shader's, tests/test_refshader_cpu.py)."""
    if _CPU_ARM:
        return _CPU_ARM
    import oracle  # the CPU baseline leg is one of the two places allowed to execute oracle/
    scene, cam, u = build_scene(rt, name)
    orc = oracle.OracleScene.from_scene(scene)
    W, H = WORKLOADS[name]["width"], WORKLOADS[name]["height"]
    region, spp = cpu_region(W, H)
    uu = u.copy()
    uu["numRaysPerPixel"] = spp
    _CPU_ARM.update(orc=orc, u=uu, region=region, spp=spp, shader=None, kind="port", segments=None, name=name)
    try:
        import refshader
        if refshader.available(False):
            tris, _ = orc.permuted()   # the oracle's BVH is pinned to the reference builder's (tests/test_oracle_cpu.py)
            _CPU_ARM["shader"] = refshader.Loaded(scene, spec_math=False, bvh=(orc.nodes(), tris))
            _CPU_ARM["kind"] = "reference"
            cn = oracle.OrcCounters()
            for f in range(CPU_SAMPLE["frames"]):
                uu["frameIndex"] = f
                orc.render_frame(uu, rng_mode=rt.RNG_REF_PCG, region=region, counters=cn)
            _CPU_ARM["segments"] = int(cn.segments)
    except Exception as e:  # a missing or stale harness must not take the bench down
        print(f"bench.py: reference shader harness unavailable ({e}); timing the oracle port", file=sys.stderr)
        _CPU_ARM.update(shader=None, kind="port", segments=None)
    return _CPU_ARM


def cpu_sample(rt, name, threads=0):
    """One bounded CPU sample of the workload: a centred crop of its image at reduced spp (throughput in Mrays/s
    does not depend on spp).  Returns (Mrays/s, seconds, segments, threads)."""
    import oracle
    arm = cpu_arm(rt, name)
    uu, region = arm["u"], arm["region"]
    nthreads = threads if threads > 0 else (os.cpu_count() or 1)
    if arm["shader"] is not None:
        t0 = time.perf_counter()
        for f in range(CPU_SAMPLE["frames"]):
            uu["frameIndex"] = f
            arm["shader"].render(uu, region=region, threads=threads)
        dt = time.perf_counter() - t0
        return arm["segments"] / dt * 1e-6, dt, arm["segments"], nthreads
    cn = oracle.OrcCounters()
    t0 = time.perf_counter()
    for f in range(CPU_SAMPLE["frames"]):
        uu["frameIndex"] = f
        arm["orc"].render_frame(uu, rng_mode=rt.RNG_PHILOX, threads=threads, region=region, counters=cn)
    dt = time.perf_counter() - t0
    return cn.segments / dt * 1e-6, dt, int(cn.segments), nthreads


def sample_text(name):
    wl = WORKLOADS[name]
    (x0, y0, x1, y1), spp = cpu_region(wl["width"], wl["height"])
    base = (f"centred {x1 - x0}x{y1 - y0} crop of the {wl['width']}x{wl['height']} image of the same scene and camera, "
            f"{CPU_SAMPLE['frames']} frame x {spp} spp, depth {wl['max_bounce']}, ")
    if _CPU_ARM.get("kind") == "reference":
        return base + ("the reference's own compute.glsl compiled for the CPU (glsl2cpp.py + glm, g++ -O2, libm) over the "
                       "reference's BVH (BVH.h), the shader's PCG stream, std::thread over rows; segments counted by the oracle "
                       "on the identical frame")
    return base + "Philox, oracle port of compute.glsl with the reference's own BVH (BVH.h), std::thread over rows"


def run_reference(args, rt):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = args.workload
    vals, secs = [], []
    nthreads = os.cpu_count() or 1
    for i in range(args.warmup + args.steps):
        v, dt, segs, nthreads = cpu_sample(rt, name)
        if i >= args.warmup:
            vals.append(v); secs.append(dt)
    value = float(np.mean(vals))
    frames_total = args.frames if args.frames > 0 else WORKLOADS[name]["frames"]
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(secs)) * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(name, frames_total, args.gpus, args.split),
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": nthreads, "kind": _CPU_ARM.get("kind", "port"),
                         "sample": sample_text(name)},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ roofline
def load_traffic(name):
    """dram__bytes per segment of k_extend, measured with ncu over every k_extend launch of one screenshot of this
    workload (tools/extend_traffic.sh -> profiles/extend_traffic.json: per workload the bytes, the kernel's git hash,
    the date and the raw CSV)."""
    try:
        t = json.load(open(os.path.join(REPO, "profiles", "extend_traffic.json")))
        e = t.get(name)
        return e if isinstance(e, dict) else None
    except Exception:
        return None


def extend_roofline(c, ci, ceil, name, bvh_bytes, ms_total, clocks, width_of_tree):
    """SURVEY.md §8d: per segment, bytes = n_node*node_bytes + n_tri*48 + 96 and flops = n_box*24 + n_tri*56 (a
    4-wide visit tests four boxes: 96 flops, the survey's 48 per two-box binary visit); t_roof = max over the
    ceilings that can bind; frac = t_roof / t_measured for the average k_extend launch of the timed region."""
    seg_i = max(ci["segments"], 1)
    n_node, n_tri = ci["node_visits"] / seg_i, ci["tri_tests"] / seg_i
    node_bytes = 64 if width_of_tree == 4 else 32
    boxes_per_visit = 4 if width_of_tree == 4 else 2
    bvh_b = n_node * node_bytes + n_tri * 48
    path_b = 96.0
    flops = n_node * boxes_per_visit * 24 + n_tri * 56
    launches = max(c["extend_launches"], 1)
    seg_per_launch = c["segments"] / launches
    t_meas = c["extend_ms"] * 1e-3 / launches
    hbm_peak, hbm_src = measured_peaks()
    l2_resident = bvh_bytes < 100e6
    g = (ceil or {}).get("gather_gbs", {})
    tname = "8MB" if l2_resident else "1GB"
    gather_peak = g.get(f"{tname}_{node_bytes}B_independent")
    fp32_peak = (ceil or {}).get("issue_tops", {}).get("fadd_fmul")
    fp32_src = "measured now (tools/microbench.cu, FADD/FMUL issue, non-FMA)"
    if not fp32_peak or fp32_peak <= 0:
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        fp32_peak, fp32_src = 148 * 128 * sm_mhz * 1e6 * 1e-12, "estimate 148 SM x 128 lanes x SM clock"
    tr = load_traffic(name)
    dram_b = tr.get("dram_bytes_per_segment") if tr else None
    t = {}
    # HBM: the path records always stream through HBM; the BVH bytes only when the BVH cannot live in L2 (then ALL of
    # them are charged to HBM at the copy peak, although the top of the tree is served by L1 / L2: an upper bound on
    # the HBM time, i.e. the most demanding of the ceilings that can be written down without a cache model)
    t["hbm"] = (path_b + (0.0 if l2_resident else bvh_b)) * seg_per_launch / (hbm_peak * 1e9)
    if l2_resident and gather_peak and gather_peak > 0:
        t["l2_gather"] = bvh_b * seg_per_launch / (gather_peak * 1e9)
    t["fp32"] = flops * seg_per_launch / (fp32_peak * 1e12)
    bound = max(t, key=lambda k: t[k])
    t_roof = t[bound]
    if bound == "fp32":
        achieved, peak, unit = flops * seg_per_launch / t_meas * 1e-12, fp32_peak, "TFLOP/s"
    elif bound == "hbm":
        achieved, peak, unit = (path_b + (0.0 if l2_resident else bvh_b)) * seg_per_launch / t_meas * 1e-9, hbm_peak, "GB/s"
    else:
        achieved, peak, unit = bvh_b * seg_per_launch / t_meas * 1e-9, gather_peak, "GB/s"
    traffic = dram_b * seg_per_launch if dram_b is not None else None
    # for the record, not a ceiling of algorithmic bytes: the DRAM bytes ncu counted, delivered in the time measured
    # here, against what HBM delivers (a) streaming and (b) as random 64-byte gathers out of a 1 GB table
    dram = None
    if dram_b is not None and t_meas > 0:
        gbs = dram_b * seg_per_launch / t_meas * 1e-9
        hg = g.get("1GB_64B_independent")
        dram = {"bytes_per_segment": dram_b, "gbs": gbs, "frac_of_hbm_copy_peak": gbs / hbm_peak,
                "frac_of_hbm_random_gather_peak": (gbs / hg) if hg else None, "hbm_random_gather_gbs": hg,
                "algorithmic_bytes_served_on_chip": 1.0 - min(1.0, dram_b / (bvh_b + path_b))}
    return {
        "kernel": "k_extend", "bound": bound, "achieved": achieved, "peak": peak, "unit": unit,
        "frac": t_roof / t_meas if t_meas > 0 else None, "traffic": traffic,
        "traffic_source": tr, "dram_measured": dram,
        "t_measured_ms": t_meas * 1e3, "t_roof_ms": {k: v * 1e3 for k, v in t.items()},
        "frac_by_ceiling": {k: (v / t_meas if t_meas > 0 else None) for k, v in t.items()},
        "peaks": {"hbm_gbs": hbm_peak, "hbm_source": hbm_src, "gather_gbs": gather_peak,
                  "gather_source": f"measured now (tools/microbench.cu: random {node_bytes} B records, {tname} table, independent)",
                  "fp32_tflops": fp32_peak, "fp32_source": fp32_src},
        "node_visits_per_segment": n_node, "tri_tests_per_segment": n_tri, "node_bytes": node_bytes,
        "bvh_bytes_per_segment": bvh_b, "path_bytes_per_segment": path_b, "bytes_per_segment": bvh_b + path_b,
        "flops_per_segment": flops, "segments_per_launch": seg_per_launch,
        "extend_share_of_step": c["extend_ms"] / ms_total if ms_total else None,
        "bvh_resident_in": "L2" if l2_resident else "HBM",
        "note": "algorithmic bytes per segment = visits x node bytes + triangle tests x 48 + 96 (ray in, hit out, next ray, "
                "throughput); counts from an instrumented replay of identical rays (counter-based RNG); duration = average "
                "k_extend launch of the timed region (CUDA events on the launching stream); frac = largest t_roof / t_measured",
    }


def shade_roofline(c, ms_total):
    """Everything outside k_extend streams path records through HBM (k_raygen, k_shade, k_accumulate, k_resolve; DESIGN.md
    §5): algorithmic bytes = per segment 64 read (48 B state + 16 B hit), per surviving segment 48 written, per path
    48 written by raygen, 16 written as its contribution and 16 read back by k_accumulate — against the measured
    HBM copy peak, over the device time the library's events give that kernel class."""
    S, P = float(c["segments"]), float(c["paths"])
    if S <= 0 or c["shade_ms"] <= 0:
        return None
    total = 64.0 * S + 48.0 * (S - P) + (48.0 + 16.0 + 16.0) * P
    hbm_peak, _ = measured_peaks()
    gbs = total / (c["shade_ms"] * 1e-3) * 1e-9
    return {"kernels": "k_raygen + k_shade + k_accumulate + k_resolve", "bound": "hbm", "achieved": gbs, "peak": hbm_peak,
            "unit": "GB/s", "frac": gbs / hbm_peak, "bytes_per_segment": total / S,
            "share_of_step": c["shade_ms"] / ms_total if ms_total else None}


# ------------------------------------------------------------------------------------------------ GPU arm
class Runner:
    def __init__(self, args, rt, torch, dist, rank, local_rank, world, stream):
        self.args, self.rt, self.torch, self.dist = args, rt, torch, dist
        self.rank, self.local_rank, self.world, self.stream = rank, local_rank, world, stream

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def make_backend(self, scene, split, **kw):
        rt = self.rt
        be = rt.Backend(device=self.local_rank, rng_mode=rt.RNG_PHILOX, split_mode=split if self.world > 1 else rt.SPLIT_NONE,
                        rank=self.rank if self.world > 1 else 0, world_size=self.world, **kw)
        # The library launches on the stream it is given; torch's default stream is the legacy stream 0, which
        # rt_set_stream treats as "use the ctx's own stream", and events recorded on stream 0 would not wait for
        # that non-blocking stream.  So: one explicit side stream for library and events.
        be.set_stream(self.stream.cuda_stream)
        if self.world > 1:
            obj = [be.comm_unique_id() if self.rank == 0 else None]
            self.dist.broadcast_object_list(obj, src=0)
            be.comm_init(obj[0])
        be.upload(scene)
        return be

    def timed(self, be, u, frames, steps, warmup, sampler=None):
        torch, stream = self.torch, self.stream
        for _ in range(warmup):
            be.screenshot_device(u, frames)
        self.barrier()
        be.reset_counters()
        if sampler is not None:
            sampler.start()
        self.barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record(stream)
        for i in range(steps):
            be.screenshot_device(u, frames)
            ev[i + 1].record(stream)
        self.barrier()
        ms_total = ev[0].elapsed_time(ev[steps])
        step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
        clocks = sampler.stop() if sampler is not None else None
        c = be.counters()
        t = torch.tensor([ms_total, float(c["segments"]), float(c["kernel_launches"])], dtype=torch.float64, device="cuda")
        if self.world > 1:
            tmax = t.clone(); self.dist.all_reduce(tmax, op=self.dist.ReduceOp.MAX)
            tsum = t.clone(); self.dist.all_reduce(tsum, op=self.dist.ReduceOp.SUM)
            ms_total, segments, launches = float(tmax[0]), float(tsum[1]), float(tsum[2])
        else:
            segments, launches = float(c["segments"]), float(c["kernel_launches"])
        return dict(ms_total=ms_total, step_ms=step_ms, counters=c, segments=segments, launches=launches, clocks=clocks,
                    value=segments / (ms_total * 1e-3) * 1e-6, ms_per_step=ms_total / steps)

    def instrumented(self, scene, u):
        """node visits / triangle tests per segment from an instrumented replay of one frame (identical rays)."""
        bi = self.rt.Backend(device=self.local_rank, rng_mode=self.rt.RNG_PHILOX, instrument=True)
        bi.set_stream(self.stream.cuda_stream)
        bi.upload(scene)
        bi.screenshot_device(u, 1)
        self.torch.cuda.synchronize()
        ci = bi.counters()
        bi.close()
        return ci

    def e2e(self, be, scene, u, frames, n):
        torch = self.torch
        tris, mats, texs = scene.triangles, scene.materials, scene.textures
        ptris, _k1 = pinned_copy(torch, tris)
        pmats, _k2 = pinned_copy(torch, mats)
        ptexs = [pinned_copy(torch, t_) for t_ in texs]
        W, H = int(u["width"][0]), int(u["height"][0])
        h2d = ptris.nbytes + pmats.nbytes + sum(p[0].nbytes for p in ptexs) + 192 * frames
        d2h = W * H * 3 if self.rank == 0 else 0
        phases = {"upload": 0.0, "build": 0.0, "screenshot": 0.0}

        def step():
            t_a = time.perf_counter()
            be.set_triangles(ptris)
            be.set_materials(pmats)
            for i, (p, _) in enumerate(ptexs):
                be.set_texture(i, p)
            t_b = time.perf_counter()
            be.build()
            t_c = time.perf_counter()
            out = be.screenshot(u, frames, want_output=(self.rank == 0))
            t_d = time.perf_counter()
            phases["upload"] += t_b - t_a; phases["build"] += t_c - t_b; phases["screenshot"] += t_d - t_c
            return out

        step()
        self.barrier()
        be.reset_counters()
        for k in phases:
            phases[k] = 0.0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(self.stream)
        shot = None
        for _ in range(n):
            shot = step()
        e1.record(self.stream)
        self.barrier()
        wall = time.perf_counter() - t0
        ce = be.counters()
        te = torch.tensor([wall, float(ce["segments"])], dtype=torch.float64, device="cuda")
        if self.world > 1:
            tm = te.clone(); self.dist.all_reduce(tm, op=self.dist.ReduceOp.MAX)
            ts = te.clone(); self.dist.all_reduce(ts, op=self.dist.ReduceOp.SUM)
            wall, seg = float(tm[0]), float(ts[1])
        else:
            seg = float(ce["segments"])
        return {"value": seg / wall * 1e-6, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "seconds_per_step": wall / n, "steps": n,
                "host_phases_ms_per_step": {k: round(v / n * 1e3, 2) for k, v in phases.items()},
                "device_ms_per_step": e0.elapsed_time(e1) / n,
                "includes": "rt_scene_set_triangles/materials/texture from pinned host memory, rt_scene_build, "
                            "rt_screenshot with RGB8 readback"}, shot


def parity_gate(rt, be, scene, name, shot, frames, world):
    """No oracle here (bench.py may not use it as more than the CPU baseline): committed golden CRCs.
    (1) first-hit ids + distances of a 240x135 view — since round 2 rt_first_hit runs the TIMED traversal kernel
    (k_extend over the 4-wide tree), so a broken node step fails here; (2) the CRC of the screenshot the end-to-end
    leg just produced against the value recorded when the kernels last passed the oracle parity suite."""
    out = {}
    meta = {}
    try:
        meta = json.load(open(os.path.join(REPO, "tests", "golden", "golden.json")))
    except FileNotFoundError:
        return {"status": "golden missing"}
    if WORKLOADS[name]["scene"] == "sphere_cornell":
        cam_s = rt.camera_for_box(scene, 240, 135)
        us = rt.screenshot_uniforms(scene, cam_s, spp=4, max_bounce=6, env_light=False)
        tri, dst = be.first_hit(us, rt.FIRST_HIT_CENTRE)
        ok = (zlib.crc32(tri.tobytes()) & 0xffffffff) == meta["config2_first_hit_240x135_crc"] and \
             (zlib.crc32(dst.tobytes()) & 0xffffffff) == meta["config2_first_hit_240x135_dst_crc"]
        out["first_hit_240x135_through_k_extend"] = "PASS" if ok else "FAIL"
        if not ok:
            raise SystemExit("bench.py: parity gate failed — first-hit ids/dst differ from tests/golden/golden.json")
    if shot is not None:
        crc = int(zlib.crc32(shot.tobytes()) & 0xffffffff)
        want = meta.get("bench_screenshot_crc", {}).get(f"{name}_{frames}f")
        out["screenshot_crc"] = crc
        out["screenshot_crc_golden"] = want
        out["screenshot"] = "unpinned (no golden for this workload / frame count)" if want is None else \
            ("PASS" if want == crc else "FAIL")
        if want is not None and want != crc:
            raise SystemExit(f"bench.py: parity gate failed — screenshot CRC {crc} != golden {want} ({name}, {frames} frames)")
    return out


def side_block(R, rt, name, frames, steps, warmup, ceil):
    """A second workload measured for the record at N = 1 (config 2 / config 4): resident throughput, roofline."""
    scene, cam, u = build_scene(rt, name)
    be = R.make_backend(scene, rt.SPLIT_NONE, kernel_timing=True)
    m = R.timed(be, u, frames, steps, warmup)
    c = m["counters"]
    shot = be.screenshot(u, frames)
    gate = parity_gate(rt, be, scene, name, shot, frames, 1)
    be.close()
    ci = R.instrumented(scene, u)
    roof = extend_roofline(c, ci, ceil, name, c["bvh_bytes"], m["ms_total"], None, c["bvh_width"])
    wl = WORKLOADS[name]
    return {"workload": wl["text"], "frames_timed": frames, "frames_of_config": wl["frames"],
            "value": m["value"], "unit": "Mrays/s", "ms_per_step": m["ms_per_step"], "steps": steps, "warmup": warmup,
            "seconds_per_full_screenshot": m["ms_per_step"] * 1e-3 * wl["frames"] / frames,
            "roofline": roof, "shade_roofline": shade_roofline(c, m["ms_total"]), "parity_gate": gate,
            "bvh": {"build_ms": c["build_ms"], "nodes": c["bvh_nodes"], "bytes": c["bvh_bytes"], "depth": c["bvh_depth"],
                    "width": c["bvh_width"], "stack_need": c["bvh_stack_need"], "build_rounds": c["bvh_build_rounds"]}}


def run_gpu(args, rt):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the CUDA backend is the product, there is no CPU fallback "
                         "(use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    R = Runner(args, rt, torch, dist, rank, local_rank, world, stream)

    name = args.workload
    wl = WORKLOADS[name]
    scene, cam, u = build_scene(rt, name)
    frames = args.frames if args.frames > 0 else wl["frames"]   # TOTAL frames of the job, whatever the GPU count
    split = rt.SPLIT_TILES if args.split == "tiles" else rt.SPLIT_FRAMES
    be = R.make_backend(scene, split, kernel_timing=True)

    ceil = None
    if rank == 0 and not args.no_microbench:
        ceil = microbench(be.counters().get("extend_blocks_per_sm", 9) or 9)

    sampler = ClockSampler(local_rank) if (rank == 0 and not os.environ.get("RT_BENCH_NO_CLOCKS")) else None
    m = R.timed(be, u, frames, args.steps, args.warmup, sampler)
    c = m["counters"]
    if args.dump_outputs and rank == 0:   # the last timed step's image, still on the device
        dump_outputs(args.dump_outputs, be.screenshot_fetch())
    e2e, shot = R.e2e(be, scene, u, frames, max(1, min(args.steps, 2)))
    gate = parity_gate(rt, be, scene, name, shot, frames, world) if rank == 0 else None

    roof = cpu = None
    blocks = {}
    if rank == 0:
        ci = R.instrumented(scene, u)
        roof = extend_roofline(c, ci, ceil, name, c["bvh_bytes"], m["ms_total"] if world == 1 else None, m["clocks"], c["bvh_width"])
    if rank == 0 and world == 1 and not args.no_cpu:
        v, dt, segs, nthreads = cpu_sample(rt, name)
        port = None
        if _CPU_ARM.get("kind") == "reference":   # for the record: the oracle port on the same crop (Philox), same threads
            import oracle
            cn = oracle.OrcCounters()
            t0 = time.perf_counter()
            _CPU_ARM["orc"].render_frame(_CPU_ARM["u"], rng_mode=rt.RNG_PHILOX, region=_CPU_ARM["region"], counters=cn)
            port = {"value": cn.segments / (time.perf_counter() - t0) * 1e-6, "unit": "Mrays/s", "kind": "port"}
        cpu = {"value": v, "unit": "Mrays/s", "cores": nthreads, "kind": _CPU_ARM.get("kind", "port"), "sample": sample_text(name),
               "oracle_port": port, "seconds": dt, "segments": segs}
    be.close()
    if rank == 0 and world == 1 and name == "4k" and not args.no_side:
        for side, fr in (("config2", 4), ("config4", 2)):
            try:
                blocks[side] = side_block(R, rt, side, fr, 3 if side == "config2" else 2, 2 if side == "config2" else 1, ceil)
            except SystemExit:
                raise
            except Exception as e:  # the side blocks never take the contract line down
                blocks[side] = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": "Mrays/s", "value": m["value"], "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(name, frames, world, args.split),
            "seconds_per_screenshot": m["ms_per_step"] * 1e-3, "step_ms": [round(x, 2) for x in m["step_ms"]],
            "segments_per_step": m["segments"] / args.steps,
            "e2e": e2e, "gpu_launches": int(m["launches"]),
            "roofline": roof, "shade_roofline": shade_roofline(c, m["ms_total"]) if world == 1 else None,
            "ceilings": ceil, "cpu_baseline": cpu, "clocks": m["clocks"], "parity_gate": gate,
            "bvh": {"build_ms": c["build_ms"], "nodes": c["bvh_nodes"], "bytes": c["bvh_bytes"], "depth": c["bvh_depth"],
                    "width": c["bvh_width"], "stack_need": c["bvh_stack_need"], "build_rounds": c["bvh_build_rounds"]},
            "checksum": gate.get("screenshot_crc") if gate else None,
        }
        line.update(blocks)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3,
                    help="timed steps of the line's `value`; the e2e leg times min(steps, 2), the config2 / config4 side "
                         "blocks a fixed 3 / 2")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-side", action="store_true", help="skip the config2 / config4 blocks of the default line")
    ap.add_argument("--no-microbench", action="store_true", help="skip the ceiling microbenchmarks")
    ap.add_argument("--frames", type=int, default=0, help="TOTAL frames of the job (default: the workload's)")
    ap.add_argument("--workload", default="4k", choices=sorted(WORKLOADS),
                    help="default and contract: 4k (BASELINE config 5 at a quarter of its samples)")
    ap.add_argument("--split", default="frames", choices=["frames", "tiles"],
                    help="N > 1: frame-slice split + ncclReduce (default) or image-tile split + gather")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the screenshot of the last timed step to DIR/*.npy (see dump_outputs); GPU path only, "
                         "the reference arm renders a crop at reduced spp that no build is compared on")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed (--impl ours)")
    rt = importlib.import_module("raytracing2-fork_b200")
    if args.impl == "reference":
        run_reference(args, rt)
    else:
        run_gpu(args, rt)


if __name__ == "__main__":
    main()
