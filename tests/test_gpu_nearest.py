"""Nearest-triangle queries on CUDA tensors (Backend.query_nearest, rt_query_nearest): k_nearest against the CPU
reference's brute force (tests/nearest_oracle.py).  Every comparison is exact: identical ids and 0 ulp on dist, u, v
and the closest point.  The rule under test: with a radius r, the unbounded result if its distance is below r, else the
miss -1 / 1e38 / 0 / 0 / (0, 0, 0); a NaN, zero or negative r and a non-finite point never hit."""
import ctypes as C
import importlib

import numpy as np
import pytest

import nearest_oracle as nro

rt = importlib.import_module("raytracing2-fork_b200")
pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

MISS = np.float32(1e38)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def backend(scene, **kw):
    be = rt.Backend(device=0, **kw)
    be.upload(scene)
    return be


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def nearest(be, pts, max_dist=None):
    md = dev(max_dist) if isinstance(max_dist, np.ndarray) else max_dist
    return tuple(t.cpu().numpy() for t in be.query_nearest(dev(pts), md))


def assert_same(a, b, what):
    assert np.array_equal(a[0], b[0]), f"{what}: ids differ at {np.flatnonzero(a[0] != b[0])[:8]}"
    for k in (1, 2, 3, 4):
        assert np.array_equal(bits(a[k]), bits(b[k])), f"{what}: output {k} differs"
    assert not any(np.isnan(x).any() for x in a[1:]), f"{what}: NaN in the outputs"


def clipped(ref, r):
    """The unbounded result clipped at the radius: what a bounded query must return."""
    tri, dist, bu, bv, cp = (x.copy() for x in ref)
    keep = (tri >= 0) & (dist < np.broadcast_to(np.float32(r), dist.shape))
    tri[~keep] = -1
    dist[~keep] = MISS
    bu[~keep] = 0.0
    bv[~keep] = 0.0
    cp[~keep] = 0.0
    return tri, dist, bu, bv, cp


def mixed_radius(ref, seed):
    """Per-point radius straddling each point's distance: at it, one ulp above, half of it, uniform in (0, 2 dist),
    +inf, 0, -1, -inf and NaN, dealt round-robin."""
    rng = np.random.default_rng(seed)
    d = np.where(ref[0] >= 0, ref[1], np.float32(5.0)).astype(np.float32)
    kinds = [d, np.nextafter(d, np.float32(np.inf)), d / np.float32(2), (d * rng.uniform(0.0, 2.0, d.size)).astype(np.float32),
             np.full_like(d, np.inf), np.zeros_like(d), np.full_like(d, -1.0), np.full_like(d, -np.inf),
             np.full_like(d, np.nan)]
    return np.choose(np.arange(d.size) % len(kinds), kinds).astype(np.float32)


def scene_diag(scene):
    v = np.concatenate([scene.triangles[k][:, :3] for k in ("a", "b", "c")])
    return float(np.linalg.norm(v.max(0) - v.min(0))), v.min(0), v.max(0)


@pytest.fixture(scope="module")
def classic():
    return rt.scene_classic_cornell()


@pytest.fixture(scope="module")
def sphere_box():
    return rt.scene_textured_sphere(n_quads=40, container="cornell", tex_size=128)  # 3200 + 16 tris


def surface_points(tris, seed):
    """Exact vertices, binary32 edge midpoints and interior barycentric samples."""
    rng = np.random.default_rng(seed)
    a, b, c = (tris[k][:, :3] for k in ("a", "b", "c"))
    verts = np.concatenate([a, b, c])
    mids = ((a + b) * np.float32(0.5)).astype(np.float32)
    w = rng.dirichlet((1, 1, 1), size=len(a))
    inner = (w[:, :1] * a + w[:, 1:2] * b + w[:, 2:] * c).astype(np.float32)
    return verts.astype(np.float32), mids, inner


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scene_name", ["classic", "sphere_box"])
def test_nearest_equals_bruteforce(request, scene_name):
    scene = request.getfixturevalue(scene_name)
    be = backend(scene)
    _, lo, hi = scene_diag(scene)
    pad = (hi - lo) * 0.25
    pts = np.random.default_rng(41).uniform(lo - pad, hi + pad, size=(20000, 3)).astype(np.float32)
    ref = nro.nearest_points(scene.triangles, pts)
    assert (ref[0] >= 0).all()
    assert_same(nearest(be, pts), ref, "unbounded")
    assert_same(nearest(be, pts, float("inf")), ref, "max_dist = inf")
    be.close()


def test_far_points(classic):
    """60 to 8 000 scene sizes away: the relative shrink of the box bound."""
    be = backend(classic)
    diag, lo, hi = scene_diag(classic)
    rng = np.random.default_rng(42)
    n = 8000
    dirs = rng.normal(size=(n, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    pts = ((lo + hi) / 2 + dirs * diag * rng.uniform(60.0, 8000.0, (n, 1))).astype(np.float32)
    ref = nro.nearest_points(classic.triangles, pts)
    assert (ref[0] >= 0).all()
    assert_same(nearest(be, pts), ref, "far points")
    assert_same(nearest(be, pts, mixed_radius(ref, 43)), clipped(ref, mixed_radius(ref, 43)), "far points, radius")
    be.close()


@pytest.mark.parametrize("scene_name", ["classic", "sphere_box"])
def test_points_on_the_surface(request, scene_name):
    scene = request.getfixturevalue(scene_name)
    tris = scene.triangles
    be = backend(scene)
    verts, mids, inner = surface_points(tris, 44)
    for name, pts in (("vertices", verts), ("edge midpoints", mids), ("interior", inner)):
        ref = nro.nearest_points(tris, pts)
        assert_same(nearest(be, pts), ref, name)
        assert (ref[1] < 1e-5).all(), name
    # an exact vertex is at distance 0 from every triangle that has it, and the lowest id among them wins (or an
    # even lower triangle that the vertex also touches)
    got = nearest(be, verts)
    assert (got[1] == 0).all()
    n = len(tris)
    owner = np.arange(3 * n) % n
    first_owner = {}
    for v, o in zip(map(bytes, verts), owner):
        first_owner[v] = min(first_owner.get(v, o), o)
    assert all(g <= first_owner[bytes(v)] for g, v in zip(got[0], verts))
    be.close()


@pytest.mark.parametrize("scene_name", ["classic", "sphere_box"])
def test_radius_rule(request, scene_name):
    scene = request.getfixturevalue(scene_name)
    be = backend(scene)
    _, lo, hi = scene_diag(scene)
    pts = np.random.default_rng(45).uniform(lo - 1, hi + 1, size=(12000, 3)).astype(np.float32)
    ref = nearest(be, pts)
    r = mixed_radius(ref, 46)
    assert_same(nearest(be, pts, r), clipped(ref, r), "mixed per-point radius")
    d = np.where(ref[0] >= 0, ref[1], np.float32(5.0)).astype(np.float32)
    got = nearest(be, pts, d)
    assert (got[0] == -1).all()
    assert_same(nearest(be, pts, np.nextafter(d, np.float32(np.inf))), ref, "radius one ulp above")
    for t in (np.inf, 0.0, -1.0, -np.inf, np.nan, 0.5):
        want = clipped(ref, np.float32(t))
        assert_same(nearest(be, pts, np.full(len(pts), t, np.float32)), want, f"radius {t}")
        assert_same(nearest(be, pts, float(t)), want, f"radius {t} (float)")
    be.close()


def test_duplicate_geometry_lowest_id_wins():
    s = rt.Scene()
    red = s.add_fixed_materials()
    s.add_cube((0, 0, 0), (2, 2, 2), (0, 0, 0), red + 2)
    tris = s.triangles
    s.add_triangles(tris)
    s.add_triangles(tris[::-1])
    be = backend(s)
    pts = np.random.default_rng(47).uniform(-3, 3, size=(5000, 3)).astype(np.float32)
    ref = nro.nearest_points(s.triangles, pts)
    assert ref[0].max() < 12
    assert_same(nearest(be, pts), ref, "duplicates, unbounded")
    above = np.nextafter(ref[1], np.float32(np.inf))
    assert_same(nearest(be, pts, above), ref, "duplicates, radius one ulp above")
    assert (nearest(be, pts, ref[1].copy())[0] == -1).all()
    be.close()


def test_degenerate_triangles_in_the_scene(sphere_box):
    """Zero-length edges, collinear and coincident vertices mixed into a scene: equal to the reference, no NaN."""
    rng = np.random.default_rng(48)
    base = sphere_box.triangles
    deg = base[rng.choice(len(base), 300, replace=False)].copy()
    k = np.arange(300) % 3
    deg["b"][k == 0] = deg["a"][k == 0]                                        # zero-length edge
    deg["c"][k == 1] = deg["a"][k == 1] + np.float32(2) * (deg["b"][k == 1] - deg["a"][k == 1])  # collinear
    deg["b"][k == 2] = deg["a"][k == 2]                                        # coincident
    deg["c"][k == 2] = deg["a"][k == 2]
    s = rt.Scene()
    s.add_fixed_materials()
    mixed = np.concatenate([base[:1500], deg, base[1500:]])
    mixed["materialIndex"] = 0
    s.add_triangles(mixed)
    be = backend(s)
    _, lo, hi = scene_diag(s)
    pts = np.concatenate([rng.uniform(lo - 1, hi + 1, size=(15000, 3)),
                          deg["a"][:, :3] + rng.normal(scale=0.01, size=(300, 3))]).astype(np.float32)
    ref = nro.nearest_points(s.triangles, pts)
    assert_same(nearest(be, pts), ref, "degenerate triangles")
    assert np.isin(ref[0], np.arange(1500, 1800)).any()
    be.close()


def test_tree_width_and_builder_do_not_change_results(monkeypatch, sphere_box):
    _, lo, hi = scene_diag(sphere_box)
    pts = np.random.default_rng(49).uniform(lo - 1, hi + 1, size=(20000, 3)).astype(np.float32)
    results = {}
    for env in ({}, {"RT_BVH_WIDTH": "2"}, {"RT_BVH_BUILDER": "lbvh"}):
        monkeypatch.delenv("RT_BVH_WIDTH", raising=False)
        monkeypatch.delenv("RT_BVH_BUILDER", raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        be = backend(sphere_box)
        ref = nearest(be, pts)
        r = results.setdefault("r", mixed_radius(ref, 50))
        key = ",".join(f"{k}={v}" for k, v in env.items()) or "defaults"
        results[key] = (ref, nearest(be, pts, r), be.counters()["bvh_width"])
        be.close()
    base = results["defaults"]
    assert base[2] == 4 and results["RT_BVH_WIDTH=2"][2] == 2
    for key in ("RT_BVH_WIDTH=2", "RT_BVH_BUILDER=lbvh"):
        assert_same(results[key][0], base[0], f"{key}, unbounded")
        assert_same(results[key][1], base[1], f"{key}, mixed radius")


def test_point_counts(sphere_box):
    be = backend(sphere_box)
    _, lo, hi = scene_diag(sphere_box)
    pts = np.random.default_rng(51).uniform(lo - 1, hi + 1, size=(100003, 3)).astype(np.float32)
    ref = nro.nearest_points(sphere_box.triangles, pts)
    r = mixed_radius(ref, 52)
    for n in (0, 1, 31, 32, 33, 127, 128, 129, 100003):
        want = tuple(x[:n] for x in ref)
        assert_same(nearest(be, pts[:n]), want, f"{n} points")
        assert_same(nearest(be, pts[:n], r[:n]), clipped(want, r[:n]), f"{n} points, radius")
    be.close()


def test_single_triangle_and_empty_scene(classic):
    s = rt.Scene()
    s.add_fixed_materials()
    s.add_triangles(classic.triangles[:1])
    be = backend(s)
    pts = np.random.default_rng(53).uniform(-6, 6, size=(3000, 3)).astype(np.float32)
    ref = nro.nearest_points(s.triangles, pts)
    assert_same(nearest(be, pts), ref, "one triangle")
    r = mixed_radius(ref, 54)
    assert_same(nearest(be, pts, r), clipped(ref, r), "one triangle, radius")
    be.close()
    e = rt.Scene()
    e.add_fixed_materials()
    be = backend(e)
    got = nearest(be, pts)
    assert (got[0] == -1).all() and (got[1] == MISS).all() and not got[2].any() and not got[4].any()
    be.close()


def test_non_finite_points_miss(sphere_box):
    be = backend(sphere_box)
    _, lo, hi = scene_diag(sphere_box)
    pts = np.random.default_rng(55).uniform(lo - 1, hi + 1, size=(4000, 3)).astype(np.float32)
    ref = nearest(be, pts)
    bad = pts.copy()
    bad[0::4, 0] = np.nan
    bad[1::4, 1] = np.inf
    bad[2::4, 2] = -np.inf
    got = nearest(be, bad)
    miss = np.arange(len(pts)) % 4 != 3
    assert (got[0][miss] == -1).all() and (got[1][miss] == MISS).all() and not got[4][miss].any()
    assert_same(tuple(x[~miss] for x in got), tuple(x[~miss] for x in ref), "finite points of the same call")
    be.close()


def test_instrumented_counters(sphere_box):
    be = backend(sphere_box, instrument=True)
    _, lo, hi = scene_diag(sphere_box)
    pts = np.random.default_rng(56).uniform(lo - 1, hi + 1, size=(20000, 3)).astype(np.float32)
    be.reset_counters()
    got = be.query_nearest(dev(pts))
    c = be.counters()
    assert c["node_visits"] > 0 and c["tri_tests"] > 0
    assert c["segments"] == 0 and c["extend_launches"] == 0 and c["kernel_launches"] == 1
    assert_same(tuple(t.cpu().numpy() for t in got), nro.nearest_points(sphere_box.triangles, pts), "instrumented")
    be.close()


@pytest.mark.parametrize("side_stream", [False, True], ids=["legacy_default_stream", "side_stream"])
def test_query_is_stream_ordered_without_host_sync(sphere_box, side_stream):
    """A sleep, then an in-place write of the points, then the query, then a consumer, all on the current stream:
    correct results prove the query waited for the write; an event recorded right after the call still pending when
    it returns proves the call did not block the host."""
    be = backend(sphere_box)
    _, lo, hi = scene_diag(sphere_box)
    pts = np.random.default_rng(57).uniform(lo - 1, hi + 1, size=(50000, 3)).astype(np.float32)
    ref = nro.nearest_points(sphere_box.triangles, pts)
    r = mixed_radius(ref, 58)
    P, R = dev(pts), dev(r)
    be.query_nearest(P[:1])  # the first query binds the ctx to its stream (that may synchronise once)
    torch.cuda.synchronize()
    stream = torch.cuda.Stream() if side_stream else torch.cuda.default_stream()
    with torch.cuda.stream(stream):
        Pw = torch.zeros_like(P)
        torch.cuda._sleep(1 << 30)  # ~0.5 s of device time on this stream
        Pw.copy_(P)
        out = be.query_nearest(Pw, R)
        ev = torch.cuda.Event()
        ev.record()
        pending = not ev.query()
        hits = (out[0] >= 0).sum()  # consumer on the same stream
    torch.cuda.synchronize()
    assert pending, "the query blocked the host"
    want = clipped(ref, r)
    assert_same(tuple(t.cpu().numpy() for t in out), want, "query after an in-place write of its points")
    assert int(hits) == int((want[0] >= 0).sum())
    be.close()


def test_rejections(classic):
    be = backend(classic)
    pts = np.random.default_rng(59).uniform(-4, 4, size=(64, 3)).astype(np.float32)
    P = dev(pts)
    for args in ((torch.from_numpy(pts),),                        # CPU tensor
                 (P.double(),),                                   # float64
                 (P[:, :2].contiguous(),),                        # wrong shape
                 (P[0],),                                         # 1-D
                 (P, torch.ones(63, device="cuda")),              # max_dist of the wrong length
                 (P, torch.ones(64, device="cuda", dtype=torch.float64)),
                 (P, torch.ones(64))):                            # max_dist on the CPU
        with pytest.raises(rt.BackendError):
            be.query_nearest(*args)
    # through the C-ABI: host pointers, counts above 2^30 or below 0 (tiny valid buffers: rejected before anything is
    # read), NULL points
    L = be.L
    tri = torch.empty(64, dtype=torch.int32, device="cuda")
    dist = torch.empty(64, dtype=torch.float32, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    host = np.zeros((64, 3), np.float32)
    hp = host.ctypes.data_as(C.c_void_p)
    cases = [
        L.rt_query_nearest(be.h, hp, None, C.c_int64(64), p(tri), None, None, None, None),
        L.rt_query_nearest(be.h, p(P), hp, C.c_int64(64), p(tri), None, None, None, None),
        L.rt_query_nearest(be.h, p(P), None, C.c_int64(64), None, None, None, None, hp),
        L.rt_query_nearest(be.h, p(P), None, C.c_int64((1 << 30) + 1), p(tri), p(dist), None, None, None),
        L.rt_query_nearest(be.h, p(P), None, C.c_int64(-1), p(tri), None, None, None, None),
        L.rt_query_nearest(be.h, None, None, C.c_int64(64), p(tri), None, None, None, None),
    ]
    for i, rc in enumerate(cases):
        assert rc == 1, (i, rc)  # RT_ERR_INVALID
        with pytest.raises(rt.BackendError):
            be._chk(rc)
    assert L.rt_query_nearest(be.h, None, None, C.c_int64(0), None, None, None, None, None) == 0
    # none of that was sticky: the ctx still answers
    assert_same(nearest(be, pts), nro.nearest_points(classic.triangles, pts), "after rejected calls")
    be.close()
    nb = rt.Backend(device=0)
    with pytest.raises(rt.BackendError):
        nb.query_nearest(P)
    nb.set_triangles(classic.triangles)
    nb.set_materials(classic.materials)
    rc = nb.L.rt_query_nearest(nb.h, p(P), None, C.c_int64(64), p(tri), None, None, None, None)
    assert rc == 6  # RT_ERR_STATE
    with pytest.raises(rt.BackendError):
        nb.query_nearest(P)
    nb.close()
