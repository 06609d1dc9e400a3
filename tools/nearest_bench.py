"""Throughput of the device-resident nearest-triangle query (Backend.query_nearest) on one GPU.

Scenes (config numbers as in bench.py / BASELINE.md): config 2 (scene_textured_sphere, 100 368 triangles) and
config 4 (scene_big_sphere, 9 999 392 triangles).  Three point sets of 16 588 800 points each (199 MB of input, more
than the 126 MB of L2), in random order (sorting the points for coherence is the caller's choice and is not done here):
  (a) surface samples: a uniformly chosen triangle, a uniform barycentric point on it, offset along the triangle's
      normal by +-0.1 % of the scene diagonal;
  (b) points uniform in the scene box padded by 10 % of its extent on every side;
  (c) set (a) with max_dist = 1 % of the scene diagonal.
Before timing, a sample of every set is compared with the CPU reference's brute force (tests/nearest_oracle.py), ids
and all outputs bit for bit, and (c) with (a) clipped at the radius.  Timing: CUDA events on the query stream, warm-up
first, every timed window at least 1 s of work, the three sets alternated three times; the median and the spread
(min, max) are reported.  An instrumented replay (instrument=1) gives node visits and triangle tests per query.  The
GPU name and power limit are read in the same run (nvidia-smi, read-only query).

    python tools/nearest_bench.py --out profiles/r4_nearest_bench.json
"""
from __future__ import annotations

import argparse
import importlib
import json
import math
import os
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (REPO, os.path.join(REPO, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
rt = importlib.import_module("raytracing2-fork_b200")

N_POINTS = 1920 * 1080 * 8
MIN_WINDOW_S = 1.0
REPS = 3


def make_scene(name):
    if name == "config2":
        return rt.scene_textured_sphere(n_quads=224, container="cornell", tex_size=1024)
    return rt.scene_big_sphere(n_quads=2236)


def point_sets(torch, tris, seed):
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    a, b, c = (torch.from_numpy(np.ascontiguousarray(tris[k][:, :3])).to(dev) for k in ("a", "b", "c"))
    v = torch.cat([a, b, c])
    lo, hi = v.min(0).values, v.max(0).values
    diag = float(torch.linalg.norm(hi - lo))
    idx = torch.randint(0, a.shape[0], (N_POINTS,), generator=g, device=dev)
    r1 = torch.rand(N_POINTS, 1, generator=g, device=dev)
    r2 = torch.rand(N_POINTS, 1, generator=g, device=dev)
    s = r1.sqrt()
    ta, tb, tc = a[idx], b[idx], c[idx]
    surf = ta * (1 - s) + tb * (s * (1 - r2)) + tc * (s * r2)
    n = torch.nn.functional.normalize(torch.cross(tb - ta, tc - ta, dim=1), dim=1)
    sign = torch.where(torch.rand(N_POINTS, 1, generator=g, device=dev) < 0.5, -1.0, 1.0)
    pa = (surf + n * (sign * 0.001 * diag)).contiguous()
    pad = (hi - lo) * 0.1
    pb = (lo - pad + torch.rand(N_POINTS, 3, generator=g, device=dev) * (hi - lo + 2 * pad)).contiguous()
    return diag, pa, pb


def check(torch, be, tris, name, pts, radius, n_ref):
    """The first n_ref points against the CPU brute force, bit for bit."""
    import nearest_oracle as nro
    got = [t[:n_ref].cpu().numpy() for t in be.query_nearest(pts[:n_ref].contiguous(), radius)]
    want = nro.nearest_points(tris, pts[:n_ref].cpu().numpy(), radius)
    same = np.array_equal(got[0], want[0]) and all(
        np.array_equal(np.ascontiguousarray(x).view(np.uint32), np.ascontiguousarray(y).view(np.uint32))
        for x, y in zip(got[1:], want[1:]))
    if not same:
        raise SystemExit(f"nearest_bench: {name} differs from the CPU reference")
    return n_ref


def time_window(torch, stream, fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


def measure(torch, stream, variants, n):
    reps = {}
    for name, fn in variants.items():
        for _ in range(2):  # warm-up
            fn()
        torch.cuda.synchronize()
        one = time_window(torch, stream, fn, 2)
        reps[name] = max(2, int(math.ceil(MIN_WINDOW_S / max(one, 1e-6))))
    runs = {k: [] for k in variants}
    for _ in range(REPS):
        for name, fn in variants.items():
            runs[name].append(time_window(torch, stream, fn, reps[name]))
    out = {}
    for name, ts in runs.items():
        rate = sorted(n / t * 1e-6 for t in ts)
        out[name] = {"mqueries_per_s_median": rate[len(rate) // 2], "mqueries_per_s_min": rate[0],
                     "mqueries_per_s_max": rate[-1], "ms_per_call_median": sorted(ts)[len(ts) // 2] * 1e3,
                     "calls_per_window": reps[name], "window_s_min": min(ts) * reps[name]}
    return out


def run_scene(torch, name, seed, n_ref):
    scene = make_scene(name)
    tris = scene.triangles
    be = rt.Backend(device=0)
    be.upload(scene)
    stream = torch.cuda.Stream()
    be.set_stream(stream.cuda_stream)
    res = {"triangles": int(tris.size), "points_per_set": N_POINTS}
    with torch.cuda.stream(stream):
        diag, pa, pb = point_sets(torch, tris, seed)
        rc = 0.01 * diag
        res["scene_diagonal"] = diag
        res["max_dist_c"] = rc
        res["checked_against_cpu_reference"] = {
            "a": check(torch, be, tris, "a", pa, None, n_ref), "b": check(torch, be, tris, "b", pb, None, n_ref),
            "c": check(torch, be, tris, "c", pa, rc, n_ref)}
        ta, da = be.query_nearest(pa)[:2]
        tc, dc = be.query_nearest(pa, rc)[:2]
        want = torch.where((ta >= 0) & (da < rc), ta, torch.full_like(ta, -1))
        if not torch.equal(tc, want):
            raise SystemExit("nearest_bench: set (c) is not set (a) clipped at the radius")
        res["c_hit_fraction"] = float((tc >= 0).float().mean())
        rct = torch.full((N_POINTS,), rc, dtype=torch.float32, device=pa.device)
        res["timing"] = measure(torch, stream, {
            "a_surface": lambda: be.query_nearest(pa),
            "b_box": lambda: be.query_nearest(pb),
            "c_surface_radius": lambda: be.query_nearest(pa, rct)}, N_POINTS)
    torch.cuda.synchronize()
    be.close()
    bi = rt.Backend(device=0, instrument=True)
    bi.upload(scene)
    counts = {}
    for wl, (p, r) in {"a_surface": (pa, None), "b_box": (pb, None), "c_surface_radius": (pa, rct)}.items():
        bi.reset_counters()
        bi.query_nearest(p, r)
        c = bi.counters()
        counts[wl] = {"node_visits_per_query": c["node_visits"] / N_POINTS,
                      "tri_tests_per_query": c["tri_tests"] / N_POINTS}
    bi.close()
    res["instrumented"] = counts
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    ap.add_argument("--scenes", default="config2,config4")
    ap.add_argument("--ref-points", default="2000,128", help="points per set checked against the CPU brute force, per scene")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("nearest_bench: no CUDA device (the query has no CPU fallback)")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True)
    result = {"gpu": smi.stdout.strip().splitlines(), "min_window_s": MIN_WINDOW_S, "alternations": REPS,
              "point_order": "random (unsorted)"}
    refs = [int(x) for x in args.ref_points.split(",")]
    for i, name in enumerate(args.scenes.split(",")):
        result[name] = run_scene(torch, name, 2000 + 10 * i, refs[min(i, len(refs) - 1)])
        print(json.dumps({name: result[name]}), flush=True)
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
