"""CPU tests (no GPU) of the nearest-triangle reference (tests/native/nearest_oracle.cpp): its binary32
point-triangle distance against an independent float64 implementation in every Voronoi region and on degenerate
triangles, and its brute-force nearest query against a float64 argmin."""
import importlib

import numpy as np

import nearest_oracle as nro

rt = importlib.import_module("raytracing2-fork_b200")


def make_tris(a, b, c):
    t = np.zeros(len(a), dtype=rt.TRIANGLE)
    t["a"][:, :3], t["b"][:, :3], t["c"][:, :3] = a, b, c
    return t


def seg_dist64(p, s0, e):
    ee = np.einsum("...k,...k", e, e)
    t = np.where(ee > 0, np.einsum("...k,...k", p - s0, e) / np.where(ee > 0, ee, 1.0), 0.0)
    t = np.clip(t, 0.0, 1.0)
    return np.linalg.norm(p - (s0 + t[..., None] * e), axis=-1)


def ref_dist64(p, tri):
    """Distance from p to the closed triangle in float64: the plane projection if it falls inside, else the nearest
    of the three edges.  The triangle is the one the GPU stores: a, a + (b - a), a + (c - a) with the edges in binary32."""
    a = tri["a"][..., :3].astype(np.float64)
    e0 = (tri["b"][..., :3] - tri["a"][..., :3]).astype(np.float64)   # binary32 subtraction, as stored
    e1 = (tri["c"][..., :3] - tri["a"][..., :3]).astype(np.float64)
    p = np.asarray(p, np.float64)
    ap = p - a
    d00, d01, d11 = (np.einsum("...k,...k", x, y) for x, y in ((e0, e0), (e0, e1), (e1, e1)))
    d20, d21 = np.einsum("...k,...k", ap, e0), np.einsum("...k,...k", ap, e1)
    den = d00 * d11 - d01 * d01
    ok = den > 1e-9 * d00 * d11
    sden = np.where(ok, den, 1.0)
    u = (d11 * d20 - d01 * d21) / sden
    v = (d00 * d21 - d01 * d20) / sden
    inside = ok & (u >= 0) & (v >= 0) & (u + v <= 1)
    face = np.linalg.norm(ap - u[..., None] * e0 - v[..., None] * e1, axis=-1)
    edges = np.minimum(np.minimum(seg_dist64(p, a, e0), seg_dist64(p, a, e1)), seg_dist64(p, a + e0, e1 - e0))
    return np.where(inside, np.minimum(face, edges), edges)


def check_one(p, tri, expect=None):
    d, u, v, q = nro.point_triangle(p, tri)
    assert np.isfinite(d) and np.isfinite(u) and np.isfinite(v) and np.isfinite(q).all()
    ref = ref_dist64(p, tri)
    a = tri["a"][:3].astype(np.float64)
    scale = np.linalg.norm(np.asarray(p, np.float64) - a) + np.linalg.norm(tri["b"][:3] - tri["a"][:3]) + \
        np.linalg.norm(tri["c"][:3] - tri["a"][:3])
    assert abs(float(d) - ref) <= 1e-5 * scale + 1e-30, (p, tri, d, ref)
    assert 0 <= u <= 1 and 0 <= v <= 1 and u + v <= 1 + 1e-6
    # the reported point is the one at the reported distance
    assert abs(np.linalg.norm(q.astype(np.float64) - np.asarray(p, np.float64)) - float(d)) <= 1e-5 * scale + 1e-30
    if expect is not None:
        region = ("A" if (u, v) == (0, 0) else "B" if (u, v) == (1, 0) else "C" if (u, v) == (0, 1) else
                  "AB" if v == 0 else "AC" if u == 0 else "BC" if u + v >= 1 - 1e-6 else "face")
        assert region == expect, (region, expect, u, v)
    return d


def test_point_triangle_every_voronoi_region():
    rng = np.random.default_rng(1)
    counts = dict.fromkeys(("A", "B", "C", "AB", "AC", "BC", "face"), 0)
    for _ in range(300):
        while True:
            V = rng.uniform(-5, 5, (3, 3)).astype(np.float32)
            e0, e1 = (V[1] - V[0]).astype(np.float64), (V[2] - V[0]).astype(np.float64)
            n = np.cross(e0, e1)
            lens = [np.linalg.norm(e0), np.linalg.norm(e1), np.linalg.norm(e1 - e0)]
            angles_ok = all(np.dot(V[(k + 1) % 3] - V[k], V[(k + 2) % 3] - V[k]) > 0.2 * lens[0] * lens[1] * 0.1
                            for k in range(3))
            if np.linalg.norm(n) > 0.3 * max(lens) ** 2 and angles_ok:   # well shaped, acute: regions are clean
                break
        tri = make_tris(V[0:1], V[1:2], V[2:3])[0]
        n = n / np.linalg.norm(n)
        c = V.astype(np.float64).mean(axis=0)
        h = rng.uniform(-2, 2)
        # vertex regions: outward from the centroid past the vertex
        for k, name in enumerate("ABC"):
            p = V[k] + (V[k] - c) * rng.uniform(0.2, 2.0) + n * h
            check_one(p.astype(np.float32), tri, name)
            counts[name] += 1
        # edge regions: from the midpoint, outward in the plane, perpendicular to the edge
        for (i, j), name in (((0, 1), "AB"), ((0, 2), "AC"), ((1, 2), "BC")):
            e = (V[j] - V[i]).astype(np.float64)
            m = V[i] + e * rng.uniform(0.2, 0.8)
            out = np.cross(e, n)
            out = out if np.dot(out, m - c) > 0 else -out
            p = m + out / np.linalg.norm(out) * rng.uniform(0.1, 2.0) + n * h
            check_one(p.astype(np.float32), tri, name)
            counts[name] += 1
        w = rng.dirichlet((2, 2, 2))
        p = w @ V.astype(np.float64) + n * h
        check_one(p.astype(np.float32), tri, "face")
        counts["face"] += 1
    assert min(counts.values()) == 300


def test_point_triangle_random_points_and_triangles():
    rng = np.random.default_rng(2)
    for _ in range(3000):
        V = rng.uniform(-10, 10, (3, 3)).astype(np.float32)
        tri = make_tris(V[0:1], V[1:2], V[2:3])[0]
        check_one(rng.uniform(-20, 20, 3).astype(np.float32), tri)


def test_point_triangle_degenerate_triangles():
    """Zero-length edges, collinear and coincident vertices: never NaN, the true distance up to rounding."""
    rng = np.random.default_rng(3)
    for _ in range(2000):
        a, b = rng.uniform(-5, 5, (2, 3)).astype(np.float32)
        t = np.float32(rng.uniform(-1.5, 2.5))
        col = (a + t * (b - a)).astype(np.float32)
        for V in ((a, a, b), (a, b, a), (b, a, a), (a, b, col), (col, a, b), (a, col, b), (a, a, a)):
            tri = make_tris(*[np.asarray(x)[None] for x in V])[0]
            for p in (rng.uniform(-8, 8, 3), a, b, (a + b) / 2, col):
                check_one(np.asarray(p, np.float32), tri)


def test_point_on_the_triangle_is_at_distance_zero():
    rng = np.random.default_rng(4)
    for _ in range(200):
        V = rng.uniform(-5, 5, (3, 3)).astype(np.float32)
        tri = make_tris(V[0:1], V[1:2], V[2:3])[0]
        for k in range(3):
            assert nro.point_triangle(V[k], tri)[0] == 0.0


def test_brute_force_agrees_with_float64_argmin():
    rng = np.random.default_rng(5)
    n, m = 300, 2000
    centres = rng.uniform(-10, 10, (n, 1, 3))
    V = (centres + rng.normal(scale=1.0, size=(n, 3, 3))).astype(np.float32)
    V[::17, 1] = V[::17, 0]                         # some degenerate ones
    tris = make_tris(V[:, 0], V[:, 1], V[:, 2])
    pts = rng.uniform(-13, 13, (m, 3)).astype(np.float32)
    tri, dist, bu, bv, closest = nro.nearest_points(tris, pts)
    D = ref_dist64(pts[:, None, :], tris[None, :])  # (m, n)
    order = np.argsort(D, axis=1)
    best, second = D[np.arange(m), order[:, 0]], D[np.arange(m), order[:, 1]]
    clear = second - best > 1e-4 * (1 + best)      # near-ties may go either way in binary32
    assert clear.mean() > 0.95
    assert np.array_equal(tri[clear], order[clear, 0])
    assert np.allclose(dist, best, rtol=1e-5, atol=1e-5)
    assert not np.isnan(dist).any() and not np.isnan(closest).any()
    # the outputs are those of the point-triangle function for the chosen triangle
    for i in range(0, m, 97):
        d, u, v, q = nro.point_triangle(pts[i], tris[tri[i]])
        assert (d, u, v) == (dist[i], bu[i], bv[i]) and np.array_equal(q, closest[i])


def test_brute_force_radius_and_miss_rules():
    rng = np.random.default_rng(6)
    V = rng.uniform(-3, 3, (50, 3, 3)).astype(np.float32)
    tris = make_tris(V[:, 0], V[:, 1], V[:, 2])
    pts = rng.uniform(-5, 5, (400, 3)).astype(np.float32)
    ref = nro.nearest_points(tris, pts)
    d = ref[1]
    for r, hit in ((d, False), (np.nextafter(d, np.float32(np.inf)), True), (np.full_like(d, np.inf), True),
                   (np.zeros_like(d), False), (np.full_like(d, -1.0), False), (np.full_like(d, np.nan), False)):
        got = nro.nearest_points(tris, pts, r)
        if hit:
            assert all(np.array_equal(x, y) for x, y in zip(got, ref))
        else:
            assert (got[0] == -1).all() and (got[1] == np.float32(1e38)).all()
            assert not got[2].any() and not got[3].any() and not got[4].any()
    bad = pts.copy()
    bad[::3, 1] = np.nan
    bad[1::3, 2] = -np.inf
    got = nro.nearest_points(tris, bad)
    assert (got[0][::3] == -1).all() and (got[0][1::3] == -1).all()
    assert np.array_equal(got[0][2::3], ref[0][2::3])
    # an empty scene: every point misses
    got = nro.nearest_points(tris[:0], pts)
    assert (got[0] == -1).all() and (got[1] == np.float32(1e38)).all()
