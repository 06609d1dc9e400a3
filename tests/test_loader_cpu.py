"""CPU tests for the OBJ + MTL + texture loader (host/rt_loader.cpp): against the reference's own
getTrianglesData_ (mesh.h:279-613) run through oracle/_ref/ref_host on the models the reference ships,
and the PNG decoder against Pillow on generated files of every colour type."""
import ctypes as C
import importlib
import io
import os

import numpy as np
import pytest

import oracle

rt = importlib.import_module("raytracing2-fork_b200")
DATA = os.path.join(os.environ.get("RT_REFERENCE", ""), "RayTracing", "Data")   # RT_REFERENCE: a reference checkout
needs_ref = pytest.mark.skipif(not (oracle.have_ref_host() and os.environ.get("RT_REFERENCE") and os.path.isdir(DATA)),
                               reason="needs a reference checkout (RT_REFERENCE) and oracle/_ref/ref_host")


@needs_ref
@pytest.mark.parametrize("model", ["campfire", "rin", "sleeping", "mccree", "autumn_kitten", "building",
                                   "robot", "plants", "toonHouse"])   # the last three carry JPEG textures
def test_loader_matches_reference_loader(tmp_path, model):
    s = rt.Scene()
    s.load_model_folder(os.path.join(DATA, model))
    import subprocess
    out = str(tmp_path / "ref.rtsc")
    subprocess.check_call([oracle.REF_HOST, "load", os.path.join(DATA, model), "none", out])
    ref = oracle.read_rtsc(out)
    t, r = s.triangles, ref["tris"]
    assert t.size == r.size > 0
    for k in ("a", "b", "c", "materialIndex"):
        assert t[k].tobytes() == r[k].tobytes(), k
    m, rm = s.materials, ref["mats"]
    assert m.size == rm.size - 5            # ref_host appends the five fixed materials (rayTracing.cpp:1268-1283)
    for k in ("color", "materialType", "textureIndex", "index", "isEdgeHighlight"):
        assert m[k].tobytes() == rm[k][: m.size].tobytes(), k
    light = m["materialType"] == rt.MAT_LIGHT
    assert np.array_equal(m["emissionStrength"][light], rm["emissionStrength"][: m.size][light])
    assert len(s.textures) == len(ref["tex"])
    for a, b in zip(s.textures, ref["tex"]):   # PNG / JPEG decode + flip identical to stb_image's, byte for byte
        assert a.shape == b.shape and np.array_equal(a, b)
    textured = np.isin(t["materialIndex"], np.where(m["materialType"] == rt.MAT_TEXTURE)[0])
    for k in ("aTex", "bTex", "cTex"):          # untextured faces carry uninitialised UVs in the reference
        assert np.array_equal(t[k][textured], r[k][textured]), k
    # the material a triangle points at is the one the reference points at
    assert t["materialIndex"].max() < m.size


@needs_ref
def test_loaded_model_in_container_matches_reference(tmp_path):
    """main()'s sequence: load, fixed materials, addCornellBox — the whole scene equals the reference's."""
    import subprocess
    model = os.path.join(DATA, "sleeping")
    out = str(tmp_path / "ref.rtsc")
    subprocess.check_call([oracle.REF_HOST, "load", model, "cornell", out])
    ref = oracle.read_rtsc(out)
    d = rt.defaults()
    s = rt.Scene()
    s.load_model_folder(model)
    red = s.add_fixed_materials()
    s.add_cornell_box(d.cornell_light_size, d.cornell_padding, red + 3, True)
    t, r = s.triangles, ref["tris"]
    assert t.size == r.size == 372 + 16
    for k in ("a", "b", "c", "materialIndex"):
        assert t[k].tobytes() == r[k].tobytes(), k
    o = oracle.OracleScene.from_scene(s)
    assert o.nodes().tobytes() == ref["nodes"].tobytes()


def test_loader_errors(tmp_path):
    s = rt.Scene()
    with pytest.raises(rt.BackendError, match="not a directory"):
        s.load_model_folder(str(tmp_path / "nope"))
    (tmp_path / "empty").mkdir()
    with pytest.raises(rt.BackendError, match="OBJ file not found"):
        s.load_model_folder(str(tmp_path / "empty"))
    quad = tmp_path / "quad"
    quad.mkdir()
    (quad / "q.obj").write_text("v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nf 1 2 3 4\n")
    with pytest.raises(rt.BackendError, match="non-triangle face"):      # mesh.h:501-506
        s.load_model_folder(str(quad))
    ok = tmp_path / "ok"
    ok.mkdir()
    (ok / "m.mtl").write_text("newmtl glow\nKd 0.5 0.25 0.125\nKe 1 2 3\nnewmtl edge\nEDGE_HIGHLIGHT\nKd 0 1 0\n")
    (ok / "t.obj").write_text("mtllib m.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 0 1\nusemtl glow\nf 1/1 2/2 3/3\n"
                              "usemtl edge\nf 1//1 3//1 2//1\nusemtl glow\nf 3 2 1\n")
    s2 = rt.Scene()
    s2.load_model_folder(str(ok))
    t, m = s2.triangles, s2.materials
    assert t.size == 3 and m.size == 3                       # `_default_`, then "edge" < "glow" in std::map order
    assert m["index"].tolist() == [0, 2, 1]                   # ... while .index is MTL file order (mesh.h:369)
    assert m["materialType"][2] == rt.MAT_LIGHT and abs(m["emissionStrength"][2] - (0.299 + 2 * 0.587 + 3 * 0.114)) < 1e-6
    assert m["isEdgeHighlight"].tolist() == [0, 1, 0]
    assert t["materialIndex"].tolist() == [1, 2, 1]
    assert t["aTex"][0].tolist() == [1.0, 0.0] and t["bTex"][0].tolist() == [0.0, 1.0] and t["cTex"][0].tolist() == [0.0, 0.0]
    with pytest.raises(rt.BackendError, match="fresh scene"):
        s2.load_model_folder(str(ok))


def _decode(png_bytes):
    L = rt.host_lib()
    buf = np.frombuffer(png_bytes, dtype=np.uint8)
    w, h, ch = C.c_int32(), C.c_int32(), C.c_int32()
    rc = L.rth_decode_png(buf.ctypes.data_as(C.c_void_p), C.c_int64(buf.size), None, C.c_int64(0), C.byref(w), C.byref(h), C.byref(ch))
    assert rc == 0, L.rth_last_error()
    out = np.zeros((h.value, w.value, ch.value), np.uint8)
    rc = L.rth_decode_png(buf.ctypes.data_as(C.c_void_p), C.c_int64(buf.size), out.ctypes.data_as(C.c_void_p),
                          C.c_int64(out.size), C.byref(w), C.byref(h), C.byref(ch))
    assert rc == 0
    return out


def test_png_decoder_against_pillow():
    from PIL import Image
    rng = np.random.default_rng(3)
    cases = []
    a = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    cases.append((Image.fromarray(a, "RGB"), a))
    a4 = rng.integers(0, 256, (20, 31, 4), dtype=np.uint8)
    cases.append((Image.fromarray(a4, "RGBA"), a4))
    g = rng.integers(0, 256, (19, 23), dtype=np.uint8)
    cases.append((Image.fromarray(g, "L"), g[..., None]))
    ga = rng.integers(0, 256, (11, 13, 2), dtype=np.uint8)
    cases.append((Image.fromarray(ga, "LA"), ga))
    bw = rng.integers(0, 2, (17, 29), dtype=np.uint8) * 255          # 1-bit gray scales to 0 / 255
    cases.append((Image.fromarray(bw, "L").convert("1"), bw[..., None]))
    pal = Image.fromarray(a, "RGB").quantize(colors=16)               # palette, 4 bits per index
    cases.append((pal, np.asarray(pal.convert("RGB"))))
    for img, want in cases:
        bio = io.BytesIO()
        img.save(bio, format="PNG")
        got = _decode(bio.getvalue())
        assert got.shape == want.shape, (img.mode, got.shape, want.shape)
        assert np.array_equal(got, want), img.mode
    g16 = (rng.integers(0, 65536, (9, 14)).astype(np.uint16))
    bio = io.BytesIO()
    Image.fromarray(g16, "I;16").save(bio, format="PNG")
    assert np.array_equal(_decode(bio.getvalue())[..., 0], (g16 >> 8).astype(np.uint8))   # stb keeps the high byte
    L = rt.host_lib()
    junk = np.zeros(64, np.uint8)
    assert L.rth_decode_png(junk.ctypes.data_as(C.c_void_p), C.c_int64(64), None, C.c_int64(0), None, None, None) == 1


def test_jpeg_decoder_against_pillow(tmp_path):
    """Reference-free sanity of the baseline JPEG decoder: a 4:4:4 baseline file written by Pillow decodes to
    within 2 levels of Pillow's own decode (different IDCT / colour rounding; byte-exactness is claimed and tested
    against stb_image only, through the reference loader), grey files too; subsampled and progressive files are
    rejected with an error, not decoded wrongly."""
    from PIL import Image
    rng = np.random.default_rng(9)
    base = rng.integers(0, 256, (9, 13, 3), dtype=np.uint8)
    img = np.kron(base, np.ones((8, 8, 1), dtype=np.uint8))[:70, :101]       # blocky content, odd size
    folder = tmp_path / "m"
    (folder / "textures").mkdir(parents=True)
    Image.fromarray(img, "RGB").save(folder / "textures" / "t.jpg", quality=92, subsampling=0)
    (folder / "m.mtl").write_text("newmtl a\nKd 1 1 1\nmap_Kd t.jpg\n")
    (folder / "m.obj").write_text("mtllib m.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 0 1\nusemtl a\nf 1/1 2/2 3/3\n")
    s = rt.Scene()
    s.load_model_folder(str(folder))
    got = s.textures[0][::-1]                                                # undo the loader's vertical flip
    want = np.asarray(Image.open(folder / "textures" / "t.jpg").convert("RGB"))
    assert got.shape == want.shape == (70, 101, 3)
    assert np.abs(got.astype(int) - want.astype(int)).max() <= 2
    Image.fromarray(img[..., 0], "L").save(folder / "textures" / "t.jpg", quality=90)
    s = rt.Scene()
    s.load_model_folder(str(folder))
    wantg = np.asarray(Image.open(folder / "textures" / "t.jpg"))
    assert s.textures[0].shape == (70, 101, 1) and np.abs(s.textures[0][::-1, :, 0].astype(int) - wantg.astype(int)).max() <= 2
    for kw, msg in ((dict(subsampling=2), "subsampled"), (dict(subsampling=0, progressive=True), "progressive")):
        Image.fromarray(img, "RGB").save(folder / "textures" / "t.jpg", quality=90, **kw)
        with pytest.raises(rt.BackendError, match=msg):
            rt.Scene().load_model_folder(str(folder))
