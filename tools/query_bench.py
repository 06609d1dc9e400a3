"""Throughput of the device-resident ray queries (Backend.query_closest / query_occluded) on one GPU.

Workloads (config numbers as in bench.py / BASELINE.md):
  (a) primary rays: 1920x1080 x 8 jittered camera rays per pixel, generated in torch from the screenshot uniforms
      (pixel corner + defocus disk + +-1/2 pixel jitter, as k_raygen builds them); closest and occluded, unbounded; and
      the host round trip of rt_trace_rays (numpy in / out) against rt_query_closest on the same rays;
  (b) short secondary rays: the hit points of (a), backed off by 1e-3 along the incoming ray, directions uniform on the
      hemisphere around the reversed incoming direction, tmax = 5 % of the scene diagonal; closest and occluded;
on the config-2 scene (100 368 triangles) and the config-4 scene (9 999 392 triangles).

Before timing, every ray set is checked: occluded == (closest id >= 0) & (closest dst < tmax), and on the primary
rays query_closest == rt_trace_rays (ids and distances, bit for bit).  Timing: CUDA events on the query stream, warm-up
first, every timed window at least 1 s of work, the variants of a workload alternated three times; the median and the
spread (min, max) are reported.  An instrumented replay (instrument=1, no speculation) gives node visits and triangle
tests per ray for each query.  The GPU name and power limit are read in the same run (nvidia-smi, read-only query).

    python tools/query_bench.py --out profiles/r3_query_bench.json
"""
from __future__ import annotations

import argparse
import importlib
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
rt = importlib.import_module("raytracing2-fork_b200")

W, H, SPP = 1920, 1080, 8
MIN_WINDOW_S = 1.0
REPS = 3


def scene_and_camera(name):
    if name == "config2":
        scene = rt.scene_textured_sphere(n_quads=224, container="cornell", tex_size=1024)
        cam = rt.camera_for_box(scene, W, H)
    else:
        scene = rt.scene_big_sphere(n_quads=2236)
        cam = rt.make_camera(W, H, (0.0, 0.0, 15.5))
    u = rt.screenshot_uniforms(scene, cam, spp=SPP, max_bounce=8, env_light=False)
    return scene, u


def primary_rays(torch, u, seed):
    """W x H x SPP camera rays: pixel-corner NDC, a point on the defocus disk, +-1/2 pixel jitter (k_raygen's recipe
    with torch's generator instead of the path tracer's streams)."""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    f = lambda k: torch.tensor(np.asarray(u[k][0][:3], np.float32), device=dev)  # noqa: E731
    cam, vf, vr, vu = f("cameraPos"), f("viewportFront"), f("viewportRight"), f("viewportUp")
    pr, pu, dr, du = f("pixelRight"), f("pixelUp"), f("defocusDiskRight"), f("defocusDiskUp")
    ty, tx = torch.meshgrid(torch.arange(H, device=dev), torch.arange(W, device=dev), indexing="ij")
    x = ((tx * 2 - W).float() / W).reshape(-1, 1).repeat_interleave(SPP, 0)
    y = ((ty * 2 - H).float() / H).reshape(-1, 1).repeat_interleave(SPP, 0)
    n = x.shape[0]
    end = cam + vf + vr * x + vu * y
    a = torch.rand(n, 1, generator=g, device=dev) * (2 * math.pi)
    o = cam + dr * torch.cos(a) + du * torch.sin(a)
    jr = torch.rand(n, 1, generator=g, device=dev) - 0.5
    ju = torch.rand(n, 1, generator=g, device=dev) - 0.5
    d = torch.nn.functional.normalize(end + pr * jr + pu * ju - o, dim=1)
    return o.contiguous(), d.contiguous()


def secondary_rays(torch, o, d, tri, dst, diag, seed):
    """From the hits of (o, d): origin = hit point backed off by 1e-3 along the ray, direction uniform on the
    hemisphere around -d, tmax = 5 % of the scene diagonal."""
    g = torch.Generator(device=o.device).manual_seed(seed)
    hit = tri >= 0
    oh, dh, th = o[hit], d[hit], dst[hit].unsqueeze(1)
    org = oh + dh * (th - 1e-3)
    v = torch.nn.functional.normalize(torch.randn(oh.shape, generator=g, device=o.device), dim=1)
    v = torch.where(((v * dh).sum(1, keepdim=True) > 0), -v, v)  # the hemisphere facing back along the ray
    return org.contiguous(), v.contiguous(), float(0.05 * diag)


def check(torch, be, o, d, tmax):
    tri, dst, _, _ = be.query_closest(o, d, tmax)
    occ = be.query_occluded(o, d, tmax)
    lim = math.inf if tmax is None else tmax
    want = (tri >= 0) & (dst < lim)
    bad = int((occ != want).sum())
    if bad:
        raise SystemExit(f"query_bench: occluded disagrees with the closest hit on {bad} rays")
    return tri, dst


def time_window(torch, stream, fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


def measure(torch, stream, variants, n_rays):
    """variants: name -> callable.  Each is sized to >= 1 s per window, then the variants alternate REPS times."""
    reps = {}
    for name, fn in variants.items():
        for _ in range(2):  # warm-up
            fn()
        torch.cuda.synchronize()
        one = time_window(torch, stream, fn, 3)
        reps[name] = max(3, int(math.ceil(MIN_WINDOW_S / max(one, 1e-6))))
    runs = {k: [] for k in variants}
    for _ in range(REPS):
        for name, fn in variants.items():
            runs[name].append(time_window(torch, stream, fn, reps[name]))
    out = {}
    for name, ts in runs.items():
        gr = sorted(n_rays / t * 1e-9 for t in ts)
        out[name] = {"grays_per_s_median": gr[len(gr) // 2], "grays_per_s_min": gr[0], "grays_per_s_max": gr[-1],
                     "ms_per_call_median": sorted(ts)[len(ts) // 2] * 1e3, "calls_per_window": reps[name],
                     "window_s_min": min(ts) * reps[name]}
    return out


def host_round_trip(torch, be, stream, o, d, n_rays):
    """rt_trace_rays from numpy (its copies and the synchronisation it ends with) against rt_query_closest on the same
    rays already on the device; the host leg is timed with the host clock since every call ends in a synchronise."""
    on, dn = o.cpu().numpy(), d.cpu().numpy()
    ref = be.trace_rays(on, dn)  # warm-up, and the reference for the identity check
    tri, dst, _, _ = be.query_closest(o, d)
    if not (np.array_equal(tri.cpu().numpy(), ref[0]) and
            np.array_equal(dst.cpu().numpy().view(np.uint32), ref[1].view(np.uint32))):
        raise SystemExit("query_bench: query_closest differs from rt_trace_rays on the primary rays")
    t0 = time.perf_counter()
    be.trace_rays(on, dn)
    one = time.perf_counter() - t0
    reps = max(2, int(math.ceil(MIN_WINDOW_S / one)))
    host, dev = [], []
    dev_reps = None
    for _ in range(REPS):
        t0 = time.perf_counter()
        for _ in range(reps):
            be.trace_rays(on, dn)
        host.append((time.perf_counter() - t0) / reps)
        if dev_reps is None:
            one_dev = time_window(torch, stream, lambda: be.query_closest(o, d), 3)
            dev_reps = max(3, int(math.ceil(MIN_WINDOW_S / one_dev)))
        dev.append(time_window(torch, stream, lambda: be.query_closest(o, d), dev_reps))
    med = lambda xs: sorted(xs)[len(xs) // 2]  # noqa: E731
    return {"rt_trace_rays_host_numpy": {"ms_per_call_median": med(host) * 1e3, "ms_min": min(host) * 1e3,
                                         "ms_max": max(host) * 1e3, "grays_per_s_median": n_rays / med(host) * 1e-9,
                                         "calls_per_window": reps},
            "rt_query_closest_device": {"ms_per_call_median": med(dev) * 1e3, "ms_min": min(dev) * 1e3,
                                        "ms_max": max(dev) * 1e3, "grays_per_s_median": n_rays / med(dev) * 1e-9,
                                        "calls_per_window": dev_reps},
            "identical_results": True}


def per_ray_counts(torch, scene, rays):
    """node visits / triangle tests per ray of each query from an instrumented replay of the same rays."""
    bi = rt.Backend(device=0, instrument=True)
    bi.upload(scene)
    out = {}
    for wl, (o, d, tm) in rays.items():
        for q, fn in (("closest", bi.query_closest), ("occluded", bi.query_occluded)):
            bi.reset_counters()
            fn(o, d, tm)
            c = bi.counters()
            out[f"{wl}_{q}"] = {"node_visits_per_ray": c["node_visits"] / o.shape[0],
                                "tri_tests_per_ray": c["tri_tests"] / o.shape[0]}
    bi.close()
    return out


def run_scene(torch, name, seed):
    scene, u = scene_and_camera(name)
    tris = scene.triangles
    pts = np.concatenate([tris["a"][:, :3], tris["b"][:, :3], tris["c"][:, :3]])
    diag = float(np.linalg.norm(pts.max(0) - pts.min(0)))
    be = rt.Backend(device=0)
    be.upload(scene)
    stream = torch.cuda.Stream()
    be.set_stream(stream.cuda_stream)
    res = {"triangles": int(tris.size), "scene_diagonal": diag}
    with torch.cuda.stream(stream):
        o, d = primary_rays(torch, u, seed)
        tri, dst = check(torch, be, o, d, None)
        so, sd, tm = secondary_rays(torch, o, d, tri, dst, diag, seed + 1)
        check(torch, be, so, sd, tm)
        n_a, n_b = o.shape[0], so.shape[0]
        res["a_primary"] = {"rays": n_a, "hit_fraction": float((tri >= 0).float().mean())}
        res["a_primary"].update(measure(torch, stream, {
            "closest": lambda: be.query_closest(o, d),
            "occluded": lambda: be.query_occluded(o, d)}, n_a))
        res["a_primary"]["host_round_trip"] = host_round_trip(torch, be, stream, o, d, n_a)
        occ_b = be.query_occluded(so, sd, tm)
        res["b_secondary"] = {"rays": n_b, "tmax": tm, "occluded_fraction": float(occ_b.float().mean())}
        res["b_secondary"].update(measure(torch, stream, {
            "closest": lambda: be.query_closest(so, sd, tm),
            "occluded": lambda: be.query_occluded(so, sd, tm)}, n_b))
    torch.cuda.synchronize()
    be.close()
    res["instrumented"] = per_ray_counts(torch, scene, {"a": (o, d, None), "b": (so, sd, tm)})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    ap.add_argument("--scenes", default="config2,config4")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("query_bench: no CUDA device (the queries have no CPU fallback)")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    result = {"gpu": smi.stdout.strip().splitlines(), "image": f"{W}x{H} x {SPP} rays per pixel",
              "min_window_s": MIN_WINDOW_S, "alternations": REPS}
    for i, name in enumerate(args.scenes.split(",")):
        result[name] = run_scene(torch, name, 1000 + 10 * i)
        print(json.dumps({name: result[name]}), flush=True)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
