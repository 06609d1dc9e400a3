"""CPU tests (no GPU): the oracle against the REAL reference host code (oracle/_ref/ref_host, compiled
from a reference checkout when RT_REFERENCE names one), against published known answers, against libm, and against the
committed golden fixtures in tests/golden/."""
import ctypes as C
import importlib
import json
import math
import os
import zlib

import numpy as np
import pytest

import oracle

rt = importlib.import_module("raytracing2-fork_b200")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
needs_ref = pytest.mark.skipif(not oracle.have_ref_host(), reason="oracle/_ref/ref_host not built (needs a reference checkout: RT_REFERENCE)")

DEFINED_MATERIAL_FIELDS = {  # fields the reference's Material::make* actually writes (mesh.h:47-102)
    rt.MAT_DIFFUSE: ["color", "materialType", "textureIndex", "isEdgeHighlight"],
    rt.MAT_LIGHT: ["color", "materialType", "textureIndex", "isEdgeHighlight", "emissionColor", "emissionStrength"],
    rt.MAT_SPECULAR: ["color", "materialType", "textureIndex", "isEdgeHighlight", "specularColor", "smoothness",
                      "specularProbability"],
    rt.MAT_TEXTURE: ["materialType", "textureIndex", "isEdgeHighlight"],
}


def tri_equal(a, b):
    return a.size == b.size and all(a[n].tobytes() == b[n].tobytes() for n in a.dtype.names if n != "pad")


# ------------------------------------------------------------------------------------------------ vs the reference
@needs_ref
def test_classic_cornell_matches_reference(tmp_path):
    ref = oracle.ref_scene("classic", None, str(tmp_path / "c.rtsc"))
    s = rt.scene_classic_cornell()
    assert s.triangles.size == 38
    assert tri_equal(s.triangles, ref["tris"])
    ours, theirs = s.materials, ref["mats"]
    assert ours.size == theirs.size == 6
    for i in range(6):
        for f in DEFINED_MATERIAL_FIELDS[int(ours["materialType"][i])]:
            assert ours[f][i].tobytes() == theirs[f][i].tobytes(), (i, f)
    o = oracle.OracleScene.from_scene(s)
    assert o.nodes().tobytes() == ref["nodes"].tobytes()  # BVH.h restated bit for bit (75 nodes)
    perm, orig = o.permuted()
    assert tri_equal(perm, ref["perm"])
    assert tri_equal(s.triangles[orig], perm)


@needs_ref
@pytest.mark.parametrize("kind", ["cornell", "mirror", "sidelit", "sky"])
def test_containers_and_bvh_match_reference(tmp_path, kind):
    base = rt.Scene()
    base.set_procedural_texture(0, 32)
    m = base.add_textured(0)
    base.add_displaced_sphere(20, (0.3, -0.2, 0.1), 3.0, 0.05, m)
    base.save(str(tmp_path / "base.rtsc"))
    ref = oracle.ref_scene(kind, str(tmp_path / "base.rtsc"), str(tmp_path / "out.rtsc"))
    d = rt.defaults()
    red = base.add_fixed_materials()
    if kind == "cornell":
        base.add_cornell_box(d.cornell_light_size, d.cornell_padding, red + 3, True)
    elif kind == "mirror":
        base.add_mirror_cornell_box(d.cornell_light_size, d.cornell_padding, red + 3, red + 4)
    elif kind == "sidelit":
        base.add_side_lit_cornell_box(d.cornell_light_size, d.cornell_padding, red + 3, red + 2, True)
    else:
        base.add_sky_light_plane(red + 3)
    assert tri_equal(base.triangles, ref["tris"])
    o = oracle.OracleScene.from_scene(base)
    assert o.nodes().tobytes() == ref["nodes"].tobytes()


@needs_ref
@pytest.mark.parametrize("params", [
    (512, 512, (0.0, 0.0, 15.5), None, None, None, None, 0.0, None),
    (1920, 1080, (1.5, 2.0, 9.0), 0.7, -0.2, 1.9, 12.0, 0.08, 3.0),
    (1000, 1000, (0.0, 5.0, 10.0), None, None, None, None, 0.0, None),
])
def test_camera_uniforms_match_reference(tmp_path, params):
    w, h, pos, hfov, pitch, yaw, focus, defocus, zoom = params
    d = rt.defaults()
    hfov = d.hfov if hfov is None else hfov
    pitch = d.pitch if pitch is None else pitch
    yaw = d.yaw if yaw is None else yaw
    focus = d.focus_distance if focus is None else focus
    zoom = d.zoom if zoom is None else zoom
    ref = oracle.ref_camera(w, h, pos, hfov, pitch, yaw, focus, defocus, zoom, str(tmp_path / "cam.bin"))
    orc = oracle.camera_uniforms(w, h, pos, hfov, pitch, yaw, focus, defocus, zoom)
    cam = rt.make_camera(w, h, pos, hfov, pitch, yaw, focus, defocus, zoom)
    host = rt.interactive_uniforms(rt.Scene(), cam)
    for k in ("cameraPos", "viewportRight", "viewportUp", "viewportFront", "pixelRight", "pixelUp",
              "defocusDiskRight", "defocusDiskUp"):
        assert orc[k].tobytes() == ref[k].tobytes(), k
        assert host[k].tobytes() == ref[k].tobytes(), k


@needs_ref
def test_rng_stream_matches_reference_host_copy(tmp_path):
    """external/math/random.h shares the integer stream with the shader; its float conversion divides in
    double and so differs from the GLSL semantics in <1 % of draws (SURVEY A.2)."""
    states, floats = oracle.ref_rng(968824447, 20000, str(tmp_path / "rng.bin"))
    L = oracle.lib()
    st = C.c_uint32(968824447)
    mism = 0
    for i in range(20000):
        v = L.orc_random(C.byref(st))
        assert st.value == states[i]
        mism += np.float32(v) != floats[i]
    assert mism < 400


def test_bvh_and_fixed_materials_match_stored_reference_output(tmp_path):
    """Without a reference checkout: tests/golden/sleeping.rtsc.gz is what the reference itself wrote for
    Data/sleeping (tests/golden/make_golden_assets.sh): its loader's triangles, the five fixed materials its main()
    appends (rayTracing.cpp:1268-1283), and the node array and triangle order of its own BVH.h over those triangles.
    The oracle's BVH restatement and the host library's fixed materials must reproduce them bit for bit."""
    import gzip
    path = tmp_path / "sleeping.rtsc"
    path.write_bytes(gzip.open(os.path.join(GOLDEN, "sleeping.rtsc.gz"), "rb").read())
    ref = oracle.read_rtsc(str(path))
    assert ref["tris"].size == 372 and ref["nodes"].size == 713
    o = oracle.OracleScene(ref["tris"], ref["mats"], ref["tex"])
    assert o.nodes().tobytes() == ref["nodes"].tobytes()
    perm, orig = o.permuted()
    assert tri_equal(perm, ref["perm"])
    assert tri_equal(ref["tris"][orig], perm)
    s = rt.Scene()
    red = s.add_fixed_materials()
    ours, theirs = s.materials[red:], ref["mats"][-5:]
    assert ours.size == 5
    for i in range(5):
        assert int(ours["materialType"][i]) == int(theirs["materialType"][i])
        for f in DEFINED_MATERIAL_FIELDS[int(ours["materialType"][i])]:
            assert ours[f][i].tobytes() == theirs[f][i].tobytes(), (i, f)


# ------------------------------------------------------------------------------------------------ known answers
def test_philox_known_answers():
    """Random123 kat_vectors for philox4x32-10."""
    L = oracle.lib()
    kats = [
        ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
        ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
        ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
         [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
    ]
    for ctr, key, want in kats:
        out = (C.c_uint32 * 4)()
        L.orc_philox4x32_10((C.c_uint32 * 4)(*ctr), (C.c_uint32 * 2)(*key), out)
        assert list(out) == want


def test_pcg_hash_first_values():
    # state update and output permutation of compute.glsl:148-154, evaluated by hand in Python ints
    state = 12345
    L = oracle.lib()
    st = C.c_uint32(state)
    for _ in range(100):
        state = (state * 747796405 + 2891336453) & 0xffffffff
        r = (((state >> ((state >> 28) + 4)) ^ state) * 277803737) & 0xffffffff
        r = ((r >> 22) ^ r) & 0xffffffff
        want = np.float32(np.float32(r) / np.float32(4294967296.0))
        assert np.float32(L.orc_random(C.byref(st))) == want
        assert st.value == state


def ulp_err(got, want):
    want32 = np.float32(want)
    ulp = np.spacing(np.abs(want32)).astype(np.float64)
    return np.abs(got.astype(np.float64) - want) / np.maximum(ulp, 1e-45)


def test_elementary_functions_close_to_libm():
    L = oracle.lib()
    x = np.linspace(0, 1, 20001, dtype=np.float32)
    cos = np.array([L.orc_cos01(float(v)) for v in x], dtype=np.float32)
    sin = np.array([L.orc_sin01(float(v)) for v in x], dtype=np.float32)
    assert ulp_err(cos, np.cos(x.astype(np.float64))).max() <= 2.0
    assert ulp_err(sin, np.sin(x.astype(np.float64))).max() <= 2.0
    e = np.linspace(-86, 0, 20001, dtype=np.float32)
    ex = np.array([L.orc_exp(float(v)) for v in e], dtype=np.float32)
    assert ulp_err(ex, np.exp(e.astype(np.float64))).max() <= 3.0
    assert L.orc_exp(-200.0) == 0.0
    a = np.linspace(-1, 1, 20001, dtype=np.float32)
    ac = np.array([L.orc_acos(float(v)) for v in a], dtype=np.float32)
    assert ulp_err(ac, np.arccos(a.astype(np.float64))).max() <= 3.0
    g = np.concatenate([np.linspace(0, 1, 20001), np.logspace(-30, 0, 2000)]).astype(np.float32)
    pg = np.array([L.orc_pow_gamma(float(v)) for v in g], dtype=np.float32)
    want = np.power(g.astype(np.float64), 1 / 2.2)
    err = ulp_err(pg, want)
    assert err[g >= 1e-3].max() <= 6.0     # the range that matters after tone mapping
    assert err[g > 0].max() <= 64.0        # |log2 x| amplifies the rounding of log2(x)/2.2 for tiny x
    assert L.orc_pow_gamma(0.0) == 0.0 and L.orc_pow_gamma(1.0) == 1.0


def test_triangle_and_box_edge_cases():
    L = oracle.lib()
    t = np.zeros(1, dtype=rt.TRIANGLE)
    t["a"] = (0, 0, 0, 0); t["b"] = (1, 0, 0, 0); t["c"] = (0, 1, 0, 0)   # normal +z
    def hit(o, d):
        dst, u, v = C.c_float(), C.c_float(), C.c_float()
        r = L.orc_ray_triangle((C.c_float * 3)(*o), (C.c_float * 3)(*d), t.ctypes.data_as(C.c_void_p),
                               C.byref(dst), C.byref(u), C.byref(v))
        return r, dst.value, u.value, v.value
    assert hit((0.25, 0.25, 1), (0, 0, -1)) == (1, 1.0, 0.25, 0.25)       # front face
    assert hit((0.25, 0.25, -1), (0, 0, 1))[0] == 0                        # back face culled (S:312)
    assert hit((0.25, 0.25, 1), (1, 0, 0))[0] == 0                         # parallel
    assert hit((0, 0, 1), (0, 0, -1))[0] == 1                              # vertex
    assert hit((0.5, 0.5, 1), (0, 0, -1))[0] == 1                          # on the hypotenuse: 1-u-v == 0
    assert hit((0.5, 0, 1), (0, 0, -1))[0] == 1                            # on an edge: v == 0
    assert hit((0.25, 0.25, 5e-7), (0, 0, -1))[0] == 0                     # dst <= 1e-6 rejected (S:319)
    assert hit((2, 2, 1), (0, 0, -1))[0] == 0
    def box(o, d, lo=(-1, -1, -1), hi=(1, 1, 1)):
        return L.orc_ray_bounds((C.c_float * 3)(*o), (C.c_float * 3)(*d), (C.c_float * 3)(*lo), (C.c_float * 3)(*hi))
    assert box((0, 0, 5), (0, 0, -1)) == 4.0
    assert box((0, 0, 5), (0, 0, 1)) == np.float32(1e38)                   # behind
    assert box((0, 0, 0), (0, 0, 1)) == -1.0                               # inside: negative entry
    assert box((5, 0, 5), (0, 0, -1)) == 4.0                               # axis with |d|<1e-6 skipped (S:394)


def test_oracle_bvh_equals_bruteforce():
    scene = rt.scene_textured_sphere(n_quads=24, container="cornell", tex_size=32)
    orc = oracle.OracleScene.from_scene(scene)
    rng = np.random.default_rng(5)
    o = rng.uniform(-3.5, 3.5, (3000, 3)).astype(np.float32)
    d = rng.normal(size=(3000, 3)); d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)
    a = orc.trace_rays(o, d, use_bvh=True)
    b = orc.trace_rays(o, d, use_bvh=False)
    for x, y in zip(a, b):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))


def test_texture_sampling_semantics():
    s = rt.Scene()
    px = np.zeros((2, 2, 3), np.uint8)
    px[0, 0] = (255, 0, 0); px[0, 1] = (0, 255, 0); px[1, 0] = (0, 0, 255); px[1, 1] = (255, 255, 255)
    s.set_texture(0, px)
    s.add_fixed_materials()
    orc = oracle.OracleScene(s.triangles, s.materials, s.textures, build=False)
    def tex(u, v):
        out = (C.c_float * 3)()
        oracle.lib().orc_sample_texture(orc.h, 0, C.c_float(u), C.c_float(v), out)
        return tuple(out)
    assert tex(0.25, 0.25) == (1.0, 0.0, 0.0)            # texel centres
    assert tex(0.75, 0.25) == (0.0, 1.0, 0.0)
    assert tex(0.25, 0.75) == (0.0, 0.0, 1.0)
    assert tex(1.25, -0.75) == (1.0, 0.0, 0.0)           # REPEAT
    assert tex(0.5, 0.25) == (0.5, 0.5, 0.0)             # bilinear halfway
    assert tex(0.0, 0.25) == (0.5, 0.5, 0.0)             # wraps across the border


def test_finalize_semantics():
    sums = np.zeros((2, 1, 3), np.uint32)
    sums[0, 0] = (10, 11, 2550)      # bottom row
    sums[1, 0] = (0, 255 * 4, 7)
    out = oracle.finalize(sums, 4)
    assert out.shape == (2, 1, 3)
    assert tuple(out[1, 0]) == (2, 2, 255)   # 10/4 and 11/4 truncate (rayTracing.cpp:249); min(255)
    assert tuple(out[0, 0]) == (0, 255, 1)   # flipped (rayTracing.cpp:253-259)


# ------------------------------------------------------------------------------------------------ goldens
def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xffffffff


def test_goldens():
    """tests/golden/*.json + *.npy were minted from this oracle by tests/golden/make_golden.py; they pin the
    oracle against silent drift (compiler, flags) and give the GPU tests a second, oracle-free anchor."""
    meta = json.load(open(os.path.join(GOLDEN, "golden.json")))
    scene = rt.scene_classic_cornell()
    orc = oracle.OracleScene.from_scene(scene)
    cam = rt.make_camera(512, 512, (0.0, 0.0, 15.5))
    u = rt.screenshot_uniforms(scene, cam, spp=64, max_bounce=8, env_light=False)
    tri, dst = orc.first_hit(u, rt.FIRST_HIT_CENTRE)
    assert crc(tri) == meta["config1_first_hit_centre_crc"]
    assert crc(dst) == meta["config1_first_hit_centre_dst_crc"]
    for mode, name in ((rt.RNG_REF_PCG, "pcg"), (rt.RNG_PHILOX, "philox")):
        tri, _ = orc.first_hit(u, rt.FIRST_HIT_SAMPLE0, rng_mode=mode)
        assert crc(tri) == meta[f"config1_first_hit_sample0_{name}_crc"]
    small = np.load(os.path.join(GOLDEN, "classic_first_hit_64.npy"))
    cam64 = rt.make_camera(64, 64, (0.0, 0.0, 15.5))
    u64 = rt.screenshot_uniforms(scene, cam64, spp=8, max_bounce=8, env_light=False)
    tri64, _ = orc.first_hit(u64, rt.FIRST_HIT_CENTRE)
    assert np.array_equal(tri64, small)
    for mode, name in ((rt.RNG_REF_PCG, "pcg"), (rt.RNG_PHILOX, "philox")):
        img = orc.render_frame(u64, rng_mode=mode)
        assert crc(img) == meta[f"classic_frame_64_{name}_crc"]
        shot, _ = orc.screenshot(u64, 2, rng_mode=mode)
        want = np.load(os.path.join(GOLDEN, f"classic_shot_64_{name}.npy"))
        assert np.array_equal(shot, want)


def test_unorm8_reciprocal_sequence_is_exact():
    """csrc/wavefront.cu::unorm8 replaces `b / 255.0f` (texel → [0,1], DESIGN.md §4.6) by q0 = b·c, r = fma(−255, q0, b),
    q = fma(r, c, q0) with c = RN(1/255).  With exact rationals: the result is the correctly rounded quotient for every
    byte, so no bit of any texel changes (the plain product b·c would be wrong for 126 of the 256 values)."""
    from fractions import Fraction
    import math

    def rn32(fr):
        if fr == 0:
            return Fraction(0)
        sign, a = (1, fr) if fr > 0 else (-1, -fr)
        e = math.floor(math.log2(float(a)))
        while Fraction(2) ** e > a:
            e -= 1
        while Fraction(2) ** (e + 1) <= a:
            e += 1
        ulp = Fraction(2) ** (e - 23)
        q = a / ulp
        n = q.numerator // q.denominator
        rem = q - n
        if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and n % 2 == 1):
            n += 1
        return sign * n * ulp

    c = rn32(Fraction(1, 255))
    assert float(c) == float(np.float32(0.003921568859368563))
    wrong_plain = 0
    for b in range(256):
        x = Fraction(b)
        q0 = rn32(x * c)
        r = rn32(x - 255 * q0)
        q = rn32(q0 + r * c)
        assert q == rn32(x / 255), b
        assert float(q) == float(np.float32(b) / np.float32(255.0))
        wrong_plain += q0 != rn32(x / 255)
    assert wrong_plain == 126


def test_rejection_test_without_sqrt():
    """k_shade evaluates the acceptance test of compute.glsl:180, `length(v) < 1`, as `dot(v, v) < 1` (no sqrt).
    The two agree for every binary32 x = dot(v, v): sqrt is monotonic and correctly rounded, sqrt(x) >= 1 for
    x >= 1, and for the largest x below 1 (1 - 2^-24) the exact root 1 - 2^-25 - 2^-51 - ... lies below the midpoint
    of (1 - 2^-24, 1) and rounds down.  Checked here on every float within 2^16 ulp of 1 and on random ones."""
    one = np.float32(1.0).view(np.uint32)
    near = (np.arange(-65536, 65537, dtype=np.int64) + int(one)).astype(np.uint32).view(np.float32)
    rng = np.random.default_rng(5)
    rnd = rng.uniform(0.0, 3.0, 2_000_000).astype(np.float32)
    for x in (near, rnd):
        assert np.array_equal(np.sqrt(x, dtype=np.float32) < np.float32(1.0), x < np.float32(1.0))


def test_signed_unit_draw_by_one_fma():
    """k_shade turns a 32-bit Philox word into a candidate component `random() * 2 - 1` (compute.glsl:153, 177-179) as
    fma(float(r), 2^-31, -1) instead of ((float(r) / 2^32) * 2) - 1.  float(r) / 2^32 and the doubling are exact scalings
    by powers of two, so both forms round the same exact value once.  Checked on every fifth binary32 in [1, 2^32] — a
    superset of the values float(r) can take — and on the edges.  The fma is emulated in binary64: x * 2^-31 is exact
    there, and the subtraction is exact for x >= 4 (the result then needs at most 53 bits); for x < 4 the result lies
    within 2^-29 of -1, far from any binary32 rounding boundary, so the second rounding cannot change it."""
    lo, hi = int(np.float32(1.0).view(np.uint32)), int(np.float32(4294967296.0).view(np.uint32))
    two31 = np.float64(2.0) ** -31
    for start in range(lo, hi + 1, 5 * (1 << 22)):
        bits = np.arange(start, min(start + 5 * (1 << 22), hi + 1), 5, dtype=np.uint32)
        x = bits.view(np.float32)
        old = (x / np.float32(4294967296.0)) * np.float32(2.0) - np.float32(1.0)
        new = (x.astype(np.float64) * two31 - 1.0).astype(np.float32)
        assert np.array_equal(old.view(np.uint32), new.view(np.uint32))
    edge = np.array([0.0, 1.0, 2.0, 3.0, 2147483648.0, 4294967040.0, 4294967296.0], np.float32)
    old = (edge / np.float32(4294967296.0)) * np.float32(2.0) - np.float32(1.0)
    new = (edge.astype(np.float64) * two31 - 1.0).astype(np.float32)
    assert np.array_equal(old.view(np.uint32), new.view(np.uint32))
