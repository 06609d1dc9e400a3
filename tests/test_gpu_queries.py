"""Ray queries on CUDA tensors (Backend.query_closest / query_occluded, rt_query_closest / rt_query_occluded): the
query variants of k_extend against rt_trace_rays and the oracle's exhaustive minimum.  Every comparison is exact
(identical ids, 0 ulp).  The two rules under test:
  - closest with tmax = the unbounded closest hit if its distance is below tmax, else the miss -1 / 1e38 / 0 / 0;
  - occluded = (closest id >= 0) & (closest dst < tmax); a NaN, zero or negative tmax never hits."""
import ctypes as C
import importlib

import numpy as np
import pytest

import oracle

rt = importlib.import_module("raytracing2-fork_b200")
pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

MISS_T = np.float32(1e38)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def random_rays(n, seed, lo, hi):
    rng = np.random.default_rng(seed)
    o = rng.uniform(lo, hi, size=(n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3))
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    return o, d


def backend(scene, **kw):
    be = rt.Backend(device=0, **kw)
    be.upload(scene)
    return be


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def closest(be, o, d, tmax=None):
    tm = dev(tmax) if isinstance(tmax, np.ndarray) else tmax
    return tuple(t.cpu().numpy() for t in be.query_closest(dev(o), dev(d), tm))


def occluded(be, o, d, tmax=None):
    tm = dev(tmax) if isinstance(tmax, np.ndarray) else tmax
    return be.query_occluded(dev(o), dev(d), tm).cpu().numpy()


def assert_same(a, b, what):
    assert np.array_equal(a[0], b[0]), f"{what}: ids differ"
    for k in (1, 2, 3):
        assert np.array_equal(bits(a[k]), bits(b[k])), f"{what}: output {k} differs"


def clipped(ref, tmax):
    """The unbounded closest hit clipped at tmax: what a bounded query must return."""
    tri, dst, bu, bv = (x.copy() for x in ref)
    keep = (tri >= 0) & (dst < np.broadcast_to(np.float32(tmax), dst.shape))
    tri[~keep] = -1
    dst[~keep] = MISS_T
    bu[~keep] = 0.0
    bv[~keep] = 0.0
    return tri, dst, bu, bv


def mixed_tmax(ref, seed):
    """Per-ray tmax straddling each ray's true distance: at it, one ulp above, half of it, uniform in (0, 2 dst),
    +inf, 0, -1, -inf and NaN, dealt round-robin."""
    tri, dst = ref[0], ref[1]
    rng = np.random.default_rng(seed)
    hitd = np.where(tri >= 0, dst, np.float32(5.0)).astype(np.float32)
    kinds = [hitd, np.nextafter(hitd, np.float32(np.inf)), hitd / np.float32(2),
             (hitd * rng.uniform(0.0, 2.0, hitd.size)).astype(np.float32),
             np.full_like(hitd, np.inf), np.zeros_like(hitd), np.full_like(hitd, -1.0),
             np.full_like(hitd, -np.inf), np.full_like(hitd, np.nan)]
    sel = np.arange(hitd.size) % len(kinds)
    return np.choose(sel, kinds).astype(np.float32)


def check_queries(be, o, d, ref, tmax, what):
    """closest(tmax) == ref clipped at tmax, occluded == (id >= 0) & (dst < tmax)."""
    got = closest(be, o, d, tmax)
    want = clipped(ref, np.float32(np.inf) if tmax is None else tmax)
    assert_same(got, want, what)
    occ = occluded(be, o, d, tmax)
    assert np.array_equal(occ, want[0] >= 0), f"{what}: occluded != closest hit below tmax"
    return got


@pytest.fixture(scope="module")
def classic():
    scene = rt.scene_classic_cornell()
    return scene, oracle.OracleScene.from_scene(scene)


@pytest.fixture(scope="module")
def sphere_box():
    scene = rt.scene_textured_sphere(n_quads=40, container="cornell", tex_size=128)  # 3200 + 16 tris
    return scene, oracle.OracleScene.from_scene(scene)


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scene_name", ["classic", "sphere_box"])
def test_closest_unbounded_equals_trace_rays_and_bruteforce(request, scene_name):
    scene, orc = request.getfixturevalue(scene_name)
    be = backend(scene)
    o, d = random_rays(20000, 21, -4.5, 4.5)
    ref = be.trace_rays(o, d)
    assert_same(ref, orc.trace_rays(o, d, use_bvh=False), "trace_rays vs brute force")
    assert_same(closest(be, o, d), ref, "query_closest(tmax=None)")
    assert_same(closest(be, o, d, float("inf")), ref, "query_closest(tmax=inf)")
    assert np.array_equal(occluded(be, o, d), ref[0] >= 0)
    assert (ref[0] >= 0).mean() > 0.9
    be.close()


def test_origins_far_outside_the_scene(classic):
    """Queries always run the widened slab test: origins thousands of scene sizes away must still find the exhaustive
    minimum (the oracle without its tree)."""
    scene, orc = classic
    be = backend(scene)
    rng = np.random.default_rng(5)
    n = 8000
    far = rng.normal(size=(n, 3))
    far = far / np.linalg.norm(far, axis=1, keepdims=True) * rng.uniform(60.0, 8000.0, (n, 1))
    target = rng.uniform(-4.5, 4.5, size=(n, 3))
    o = far.astype(np.float32)
    d = target - far
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    ref = orc.trace_rays(o, d, use_bvh=False)
    assert_same(be.trace_rays(o, d), ref, "trace_rays, far origins")
    assert_same(closest(be, o, d), ref, "query_closest, far origins")
    check_queries(be, o, d, ref, mixed_tmax(ref, 6), "far origins, mixed tmax")
    assert (ref[0] >= 0).mean() > 0.5
    be.close()


@pytest.mark.parametrize("scene_name", ["classic", "sphere_box"])
def test_tmax_straddling_the_true_distance(request, scene_name):
    scene, _ = request.getfixturevalue(scene_name)
    be = backend(scene)
    o, d = random_rays(12000, 22, -4.0, 4.0)
    ref = be.trace_rays(o, d)
    hit = ref[0] >= 0
    dst = np.where(hit, ref[1], np.float32(5.0)).astype(np.float32)
    # tmax = dst: a miss; one ulp above: the hit
    got = check_queries(be, o, d, ref, dst, "tmax = dst")
    assert (got[0] == -1).all()
    got = check_queries(be, o, d, ref, np.nextafter(dst, np.float32(np.inf)), "tmax = nextafter(dst, inf)")
    assert np.array_equal(got[0], ref[0])
    got = check_queries(be, o, d, ref, dst / np.float32(2), "tmax = dst / 2")
    assert (got[0] == -1).all()
    for t in (np.inf, 0.0, -1.0, -np.inf, np.nan):
        got = check_queries(be, o, d, ref, np.full(o.shape[0], t, np.float32), f"tmax = {t}")
        assert (got[0] >= 0).any() == (t == np.inf)
        check_queries(be, o, d, ref, float(t), f"tmax = {t} (broadcast float)")
    check_queries(be, o, d, ref, mixed_tmax(ref, 23), "mixed per-ray tmax")
    be.close()


def test_duplicate_geometry_ties_at_the_bound():
    """The construction of test_ties_resolve_to_lowest_index: every triangle three times.  With tmax one ulp above
    the distance, bestT starts AT the distance, so the first candidate is taken without the tie-break and the copies
    after it tie: the lowest id must still win.  With tmax equal to the distance the query misses."""
    s = rt.Scene()
    red = s.add_fixed_materials()
    s.add_cube((0, 0, 0), (2, 2, 2), (0, 0, 0), red + 2)
    tris = s.triangles
    s.add_triangles(tris)
    s.add_triangles(tris[::-1])
    be = backend(s)
    orc = oracle.OracleScene.from_scene(s)
    o, _ = random_rays(5000, 3, -6, 6)
    d = (-o / np.linalg.norm(o, axis=1, keepdims=True)).astype(np.float32)
    ref = orc.trace_rays(o, d, use_bvh=False)
    assert (ref[0] >= 0).mean() > 0.9 and ref[0].max() < 12  # origins inside the cube see back faces: misses
    assert_same(closest(be, o, d), ref, "duplicates, unbounded")
    above = np.nextafter(ref[1], np.float32(np.inf))
    assert_same(check_queries(be, o, d, ref, above, "duplicates, tmax just above"), ref, "duplicates, tmax just above")
    got = check_queries(be, o, d, ref, ref[1].copy(), "duplicates, tmax = dst")
    assert (got[0] == -1).all()
    be.close()


def test_tree_width_and_builder_do_not_change_query_results(monkeypatch, sphere_box):
    scene, _ = sphere_box
    o, d = random_rays(20000, 24, -4.0, 4.0)
    results = {}
    for env in ({}, {"RT_BVH_WIDTH": "2"}, {"RT_BVH_BUILDER": "lbvh"}):
        monkeypatch.delenv("RT_BVH_WIDTH", raising=False)
        monkeypatch.delenv("RT_BVH_BUILDER", raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        be = backend(scene)
        ref = be.trace_rays(o, d)
        tm = mixed_tmax(ref, 25) if not results else results["tm"]
        results.setdefault("tm", tm)
        key = ",".join(f"{k}={v}" for k, v in env.items()) or "defaults"
        results[key] = (closest(be, o, d), closest(be, o, d, tm), occluded(be, o, d, tm), be.counters()["bvh_width"])
        be.close()
    base = results["defaults"]
    assert base[3] == 4 and results["RT_BVH_WIDTH=2"][3] == 2
    for key in ("RT_BVH_WIDTH=2", "RT_BVH_BUILDER=lbvh"):
        r = results[key]
        assert_same(r[0], base[0], f"{key}, unbounded")
        assert_same(r[1], base[1], f"{key}, mixed tmax")
        assert np.array_equal(r[2], base[2]), f"{key}, occluded"


def test_ray_counts_around_warp_and_claim_sizes(sphere_box):
    scene, orc = sphere_box
    be = backend(scene)
    o, d = random_rays(100003, 26, -4.0, 4.0)
    ref = be.trace_rays(o, d)
    tm = mixed_tmax(ref, 27)
    for n in (0, 1, 31, 32, 33, 127, 128, 129, 100003):
        r = tuple(x[:n] for x in ref)
        assert_same(closest(be, o[:n], d[:n]), r, f"{n} rays, unbounded")
        check_queries(be, o[:n], d[:n], r, tm[:n], f"{n} rays, mixed tmax")
    small = orc.trace_rays(o[:4000], d[:4000], use_bvh=False)
    assert_same(tuple(x[:4000] for x in ref), small, "trace_rays vs brute force")
    be.close()


def test_single_triangle_scene(classic):
    """One triangle: the root is a leaf, no inner node exists."""
    scene, _ = classic
    s = rt.Scene()
    s.add_fixed_materials()
    s.add_triangles(scene.triangles[:1])
    be = backend(s)
    orc = oracle.OracleScene.from_scene(s)
    t = scene.triangles[0]
    centre = (t["a"][:3] + t["b"][:3] + t["c"][:3]) / 3
    o, _ = random_rays(3000, 28, -6.0, 6.0)
    d = centre[None, :] + np.random.default_rng(29).normal(scale=1.0, size=o.shape) - o
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    ref = orc.trace_rays(o, d, use_bvh=False)
    assert 0 < (ref[0] >= 0).sum() < o.shape[0]
    assert_same(be.trace_rays(o, d), ref, "trace_rays, one triangle")
    assert_same(closest(be, o, d), ref, "query_closest, one triangle")
    check_queries(be, o, d, ref, mixed_tmax(ref, 30), "one triangle, mixed tmax")
    be.close()


def test_instrumented_counters(sphere_box):
    """segments grows by the ray count per query; ANY visits and tests no more than CLOSEST on the same rays with the
    same tmax (the instrumented walk does not speculate, and ANY's walk is a prefix of CLOSEST's)."""
    scene, _ = sphere_box
    o, d = random_rays(20000, 31, -4.0, 4.0)
    for tmax in (None, 1.5):
        be = backend(scene, instrument=True)
        O, D = dev(o), dev(d)
        got = {}
        for name, fn in (("closest", be.query_closest), ("any", be.query_occluded)):
            be.reset_counters()
            fn(O, D, tmax)
            got[name] = be.counters()
            assert got[name]["segments"] == o.shape[0]
            assert got[name]["extend_launches"] == 1 and got[name]["kernel_launches"] == 2
        assert got["any"]["node_visits"] <= got["closest"]["node_visits"], (tmax, got)
        assert got["any"]["tri_tests"] <= got["closest"]["tri_tests"], (tmax, got)
        assert got["closest"]["node_visits"] > 0 and got["any"]["tri_tests"] > 0
        be.close()


@pytest.mark.parametrize("side_stream", [False, True], ids=["legacy_default_stream", "side_stream"])
def test_queries_are_stream_ordered_without_host_sync(sphere_box, side_stream):
    """A sleep, then an in-place write of the rays, then the queries, then a consumer, all on the current stream:
    correct results prove the queries waited for the write; events recorded right after each call still pending when
    it returns prove the call did not block the host."""
    scene, _ = sphere_box
    be = backend(scene)
    o, d = random_rays(50000, 32, -4.0, 4.0)
    ref = be.trace_rays(o, d)
    tm = mixed_tmax(ref, 33)
    O, D, TM = dev(o), dev(d), dev(tm)
    be.query_closest(O[:1], D[:1])  # the first query binds the ctx to its stream (that may synchronise once)
    torch.cuda.synchronize()
    stream = torch.cuda.Stream() if side_stream else torch.cuda.default_stream()
    with torch.cuda.stream(stream):
        Ow = torch.zeros_like(O)
        Dw = torch.zeros_like(D)
        Dw[:, 2] = 1.0
        torch.cuda._sleep(1 << 30)  # ~0.5 s of device time on this stream
        Ow.copy_(O)
        Dw.copy_(D)
        tri, dst, bu, bv = be.query_closest(Ow, Dw, TM)
        e1 = torch.cuda.Event()
        e1.record()
        pending1 = not e1.query()
        occ = be.query_occluded(Ow, Dw, TM)
        e2 = torch.cuda.Event()
        e2.record()
        pending2 = not e2.query()
        hits = (tri >= 0).sum()  # consumer on the same stream
        occ_copy = occ.clone()
    torch.cuda.synchronize()
    assert pending1 and pending2, "a query blocked the host"
    got = tuple(x.cpu().numpy() for x in (tri, dst, bu, bv))
    want = clipped(ref, tm)
    assert_same(got, want, "query after an in-place write of its rays")
    assert np.array_equal(occ_copy.cpu().numpy(), want[0] >= 0)
    assert int(hits) == int((want[0] >= 0).sum())
    be.close()


def test_rejections(classic):
    scene, _ = classic
    be = backend(scene)
    o, d = random_rays(64, 34, -4.0, 4.0)
    O, D = dev(o), dev(d)
    for fn in (be.query_closest, be.query_occluded):
        with pytest.raises(rt.BackendError):
            fn(torch.from_numpy(o), D)                       # CPU tensor
        with pytest.raises(rt.BackendError):
            fn(O, D.double())                                # float64
        with pytest.raises(rt.BackendError):
            fn(O[:, :2].contiguous(), D[:, :2].contiguous())  # wrong shape
        with pytest.raises(rt.BackendError):
            fn(O, D[:32])                                    # N mismatch
        with pytest.raises(rt.BackendError):
            fn(O, D, torch.ones(63, device="cuda"))          # tmax of the wrong length
        with pytest.raises(rt.BackendError):
            fn(O, D, torch.ones(64, device="cuda", dtype=torch.float64))
        with pytest.raises(rt.BackendError):
            fn(O, D, torch.ones(64))                         # tmax on the CPU
    # through the C-ABI: a host pointer, a count above 2^30 (tiny valid buffers: rejected before anything is read),
    # a negative count, a NULL output
    L = be.L
    tri = torch.empty(64, dtype=torch.int32, device="cuda")
    occ = torch.empty(64, dtype=torch.uint8, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    host = np.zeros((64, 3), np.float32)
    hp = host.ctypes.data_as(C.c_void_p)
    cases = [
        L.rt_query_closest(be.h, hp, p(D), None, C.c_int64(64), p(tri), None, None, None),
        L.rt_query_closest(be.h, p(O), p(D), None, C.c_int64(64), host.ctypes.data_as(C.c_void_p), None, None, None),
        L.rt_query_occluded(be.h, p(O), p(D), hp, C.c_int64(64), p(occ)),
        L.rt_query_occluded(be.h, p(O), p(D), None, C.c_int64(64), hp),
        L.rt_query_closest(be.h, p(O), p(D), None, C.c_int64((1 << 30) + 1), p(tri), None, None, None),
        L.rt_query_occluded(be.h, p(O), p(D), None, C.c_int64((1 << 30) + 1), p(occ)),
        L.rt_query_closest(be.h, p(O), p(D), None, C.c_int64(-1), p(tri), None, None, None),
        L.rt_query_occluded(be.h, p(O), p(D), None, C.c_int64(64), None),
        L.rt_query_closest(be.h, None, p(D), None, C.c_int64(64), p(tri), None, None, None),
    ]
    for i, rc in enumerate(cases):
        assert rc == 1, (i, rc)  # RT_ERR_INVALID
        with pytest.raises(rt.BackendError):
            be._chk(rc)
    assert L.rt_query_occluded(be.h, None, None, None, C.c_int64(0), None) == 0  # count 0: nothing to do
    # none of that was sticky: the ctx still answers
    ref = be.trace_rays(o, d)
    assert_same(closest(be, o, d), ref, "after rejected calls")
    be.close()
    # an unbuilt scene
    nb = rt.Backend(device=0)
    for fn in (nb.query_closest, nb.query_occluded):
        with pytest.raises(rt.BackendError):
            fn(O, D)
    nb.set_triangles(scene.triangles)
    nb.set_materials(scene.materials)
    with pytest.raises(rt.BackendError):
        nb.query_closest(O, D)
    nb.close()
