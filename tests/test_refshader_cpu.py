"""The oracle pinned against the reference's OWN shader source (CPU tests, no GPU).

oracle/_ref/libref_shader.so is RayTracing/Assets/Shaders/compute.glsl itself — rewritten syntactically by
oracle/glsl2cpp.py, compiled with g++ -ffp-contract=off against the reference's vendored glm 0.9.9.7, run over
the node array the reference's own BVH.h builds (oracle/_ref/ref_host).  It exists wherever `make -C oracle`
saw a reference checkout (RT_REFERENCE).  The committed
tests/golden/refshader_images.npz are its outputs; the tests below hold

  * golden == reference shader, regenerated here           (skipped without the library)
  * oracle == golden, bit for bit, every case              (always)
  * reference shader with libm's cosf/sinf/expf/acosf/powf instead of the spec'd elementary functions stays
    within a few ulp of the golden                         (skipped without the library)
"""
import json
import os
import zlib

import numpy as np
import pytest

import oracle
import refshader
import scenes

rt = scenes.rt
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = scenes.refshader_cases()


@pytest.fixture(scope="module")
def golden():
    z = np.load(os.path.join(GOLD, "refshader_images.npz"))
    meta = json.load(open(os.path.join(GOLD, "refshader.json")))
    assert sorted(z.files) == sorted(CASES) == sorted(meta)
    for k in z.files:
        assert (zlib.crc32(z[k].tobytes()) & 0xffffffff) == meta[k]["crc"]
    return z


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_equals_reference_shader_golden(golden, name):
    scene, u = CASES[name]
    img = oracle.OracleScene.from_scene(scene).render_frame(u, rng_mode=rt.RNG_REF_PCG)
    ref = golden[name]
    assert img.shape == ref.shape
    diff = bits(img) != bits(ref)
    assert not diff.any(), f"{name}: {int(diff.sum())} of {diff.size} floats differ from the reference shader"


@pytest.mark.skipif(not refshader.available(True), reason="oracle/_ref/libref_shader.so not built (needs a reference checkout: RT_REFERENCE)")
@pytest.mark.parametrize("name", sorted(CASES))
def test_golden_is_what_the_reference_shader_computes(golden, name):
    scene, u = CASES[name]
    assert np.array_equal(bits(refshader.render(scene, u, spec_math=True)), bits(golden[name]))


@pytest.mark.skipif(not refshader.available(False), reason="oracle/_ref/libref_shader_libm.so not built")
@pytest.mark.parametrize("name", sorted(CASES))
def test_libm_elementary_functions_stay_within_ulps(golden, name):
    """cos / sin / exp / acos / pow are a GL driver's in the reference; with glibc's float versions in their place
    the stored sRGB floats move by a few ulp at most (pow(x, 1/2.2) is the only one on every pixel)."""
    scene, u = CASES[name]
    img = refshader.render(scene, u, spec_math=False)
    d = np.abs(bits(img).astype(np.int64) - bits(golden[name]).astype(np.int64))
    assert d.max() <= 8, f"{name}: {d.max()} ulp"
    q = lambda x: np.floor(np.clip(x[..., :3], 0, 1) * 255.0 + 0.5)
    assert (q(img) != q(golden[name])).mean() < 1e-3   # the RGB8 blit agrees but for rounding-boundary cases


def test_translator_is_syntactic():
    """glsl2cpp.py on a probe: qualifiers dropped, float suffixes, references, swizzles, hoisted random() pair."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("glsl2cpp", os.path.join(os.path.dirname(GOLD), "..", "oracle", "glsl2cpp.py"))
    g = importlib.util.module_from_spec(spec); spec.loader.exec_module(g)
    src = """#version 430 core
layout (local_size_x = 8) in;
layout(binding = 1, std430) buffer B { Thing things[]; };
layout(binding = 3, std140) uniform U { int n; vec4 p; };
float f(inout uint s, out bool b) { return 2.0 * 1e-6 + 1.5f + p.xyz.x; }
void main()
{
    vec3 e = a + b.xyz * random(-0.5f, 0.5f, s) + c.xyz * random(-0.5f, 0.5f, s);
    switch (k)
    {
        case 0:
            vec3 d = vec3(1.0);
            break;
    }
    vec3 g = vec3(0.5);
}
"""
    out = g.translate(src)
    assert "#version" not in out and "layout" not in out and "uniform" not in out
    assert "Thing* things;" in out and "int n;" in out
    assert "float f(uint& s, bool& b)" in out
    assert "2.0f * 1e-6f + 1.5f + xyz(p).x" in out
    assert "void shader_main()" in out
    assert "vec3 d; d = vec3(1.0f);" in out and "vec3 g = vec3(0.5f);" in out
    lines = [l.strip() for l in out.split("\n")]
    i = lines.index("float _rnd0 = random(-0.5f, 0.5f, s);")
    assert lines[i + 1] == "float _rnd1 = random(-0.5f, 0.5f, s);"
    assert lines[i + 2] == "vec3 e = a + xyz(b) * _rnd0 + xyz(c) * _rnd1;"


@pytest.mark.parametrize("name", sorted(scenes.refshader_big_cases()))
def test_oracle_equals_reference_shader_at_full_size(name):
    """BASELINE config 1 at its full size (512x512, 64 spp, depth 8) and the 100 368-triangle config-2 scene: the
    oracle's frame against the CRCs the reference shader source produced (tests/golden/refshader_big.json)."""
    big = json.load(open(os.path.join(GOLD, "refshader_big.json")))[name]
    scene, u = scenes.refshader_big_cases()[name]
    img = oracle.OracleScene.from_scene(scene).render_frame(u, rng_mode=rt.RNG_REF_PCG)
    assert list(img.shape) == big["shape"]
    rows = [zlib.crc32(img[y].tobytes()) & 0xffffffff for y in range(img.shape[0])]
    bad = [y for y in range(img.shape[0]) if rows[y] != big["row_crc"][y]]
    assert not bad, f"{name}: {len(bad)} rows differ from the reference shader, first {bad[:5]}"
    assert (zlib.crc32(img.tobytes()) & 0xffffffff) == big["crc"]


_DATA = os.path.join(os.environ.get("RT_REFERENCE", ""), "RayTracing", "Data")


@pytest.mark.skipif(not (refshader.available(True) and os.environ.get("RT_REFERENCE") and os.path.isdir(_DATA)),
                    reason="needs a reference checkout (RT_REFERENCE) and its harness")
@pytest.mark.parametrize("model,container", [("robot", "cornell"), ("autumn_kitten", "none"), ("campfire", "cornell"),
                                             ("rin", "none"), ("sleeping", "cornell"), ("mccree", "none"),
                                             ("building", "none"), ("plants", "cornell"), ("toonHouse", "none")])
def test_real_assets_oracle_equals_reference_shader(model, container):
    """Shipped models through the folder loader (config 2(i): Data/robot, 25 599 triangles, three textures up to
    4096²; autumn_kitten carries the isEdgeHighlight / GLASS_HIGHLIGHT materials): oracle frame == shader frame."""
    s = rt.Scene()
    s.load_model_folder(os.path.join(_DATA, model))
    red = s.add_fixed_materials()
    d = rt.defaults()
    if container == "cornell":
        s.add_cornell_box(d.cornell_light_size, d.cornell_padding, red + 3, True)
    cam = rt.camera_for_box(s, 72, 72)
    u = rt.screenshot_uniforms(s, cam, spp=4, max_bounce=10, env_light=(container == "none"))
    img = oracle.OracleScene.from_scene(s).render_frame(u, rng_mode=rt.RNG_REF_PCG)
    ref = refshader.render(s, u, spec_math=True)
    diff = bits(img) != bits(ref)
    assert not diff.any(), f"{model}: {int(diff.sum())} of {diff.size} floats differ"
    assert np.unique(ref).size > 10


@pytest.mark.skipif(not refshader.available(True), reason="oracle/_ref/libref_shader.so not built (needs a reference checkout: RT_REFERENCE)")
@pytest.mark.parametrize("seed", range(64))
def test_fuzz_oracle_equals_reference_shader(seed):
    """Seeded random triangle soups (every material type, 1/3/4-channel non-power-of-two textures, out-of-range
    texture index, defocus, sky on/off, previews, random frameIndex): oracle frame == reference shader frame."""
    scene, u = scenes.random_scene(seed)
    img = oracle.OracleScene.from_scene(scene).render_frame(u, rng_mode=rt.RNG_REF_PCG)
    ref = refshader.render(scene, u, spec_math=True)
    diff = bits(img) != bits(ref)
    nan_both = np.isnan(img) & np.isnan(ref)
    assert not (diff & ~nan_both).any(), f"seed {seed}: {int((diff & ~nan_both).sum())} of {diff.size} floats differ"
    assert np.unique(ref[..., :3]).size > 2   # not a blank image


@pytest.mark.skipif(not refshader.available(True), reason="oracle/_ref/libref_shader.so not built (needs a reference checkout: RT_REFERENCE)")
def test_screenshot_from_reference_shader_frames():
    """screenshot() of rayTracing.cpp:184-259 rebuilt around the reference shader: frame f is one dispatch with
    frameIndex = f, read back as RGB8 (round to nearest), accumulated as float, divided by the frame count, clamped,
    truncated and flipped — written here in numpy, independently of the oracle's C++ — equals orc_screenshot, which
    the CUDA rt_screenshot is tested against."""
    scene, u = CASES["zoo_96x64_spp8_d10_env"]
    frames = 3
    loaded = refshader.Loaded(scene, spec_math=True)
    acc = np.zeros((64, 96, 3), np.float32)
    for f in range(frames):
        uf = u.copy(); uf["frameIndex"] = f
        img = loaded.render(uf)[..., :3]
        q = np.floor(np.clip(np.nan_to_num(img, nan=0.0), 0.0, 1.0) * np.float32(255.0) + np.float32(0.5)).astype(np.uint8)
        acc += q.astype(np.float32)
    avg = acc / np.float32(frames)
    out = np.minimum(avg, np.float32(255.0)).astype(np.uint8)[::-1]      # truncate, then flip to top-down
    shot, sums = oracle.OracleScene.from_scene(scene).screenshot(u, frames, rng_mode=rt.RNG_REF_PCG)
    assert np.array_equal(shot, out)
    assert np.array_equal(sums, acc.astype(np.uint32))
