"""ctypes view of oracle/_ref/libref_shader*.so: the reference's OWN compute shader source, rewritten
syntactically by oracle/glsl2cpp.py and compiled against the reference's own glm (oracle/ref_shader.cpp).
TEST INFRASTRUCTURE ONLY; present only where a reference checkout (RT_REFERENCE) was available to `make -C oracle`."""
import ctypes as C
import importlib
import os
import tempfile

import numpy as np

import oracle

rt = importlib.import_module("raytracing2-fork_b200")
REF_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref")
_libs = {}


def path(spec_math=True):
    return os.path.join(REF_DIR, "libref_shader.so" if spec_math else "libref_shader_libm.so")


def available(spec_math=True) -> bool:
    return os.path.exists(path(spec_math))


def lib(spec_math=True) -> C.CDLL:
    if spec_math not in _libs:
        L = C.CDLL(path(spec_math))
        L.refsh_set_scene.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32]
        L.refsh_set_texture.argtypes = [C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32]
        L.refsh_render.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.refsh_render_region.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int]
        assert L.refsh_spec_math() == (1 if spec_math else 0)
        _libs[spec_math] = L
    return _libs[spec_math]


def reference_bvh(scene):
    """(nodes, permuted triangles) from the REAL reference builder (BVH.h through oracle/_ref/ref_host) when it
    is there, else from the oracle's restatement of it (tests/test_oracle_cpu.py pins the two to each other)."""
    if oracle.have_ref_host():
        with tempfile.TemporaryDirectory() as d:
            scene.save(os.path.join(d, "in.rtsc"))
            out = oracle.ref_scene("none", os.path.join(d, "in.rtsc"), os.path.join(d, "out.rtsc"))
            return out["nodes"].copy(), out["perm"].copy()
    orc = oracle.OracleScene.from_scene(scene)
    tris, _ = orc.permuted()
    return orc.nodes(), tris


class Loaded:
    """A scene bound to the reference shader (reference BVH built once); render() = one dispatch."""

    def __init__(self, scene, spec_math=True, bvh=None):
        self.L = lib(spec_math)
        nodes, tris = bvh if bvh is not None else reference_bvh(scene)
        self.nodes = np.ascontiguousarray(nodes, dtype=rt.REF_NODE)
        self.tris = np.ascontiguousarray(tris, dtype=rt.TRIANGLE)
        self.mats = np.ascontiguousarray(scene.materials, dtype=rt.MATERIAL)
        self.tex = [np.ascontiguousarray(t, dtype=np.uint8) for t in scene.textures]

    def bind(self):
        L = self.L
        assert L.refsh_set_scene(self.tris.ctypes.data, self.tris.size, self.nodes.ctypes.data, self.nodes.size,
                                 self.mats.ctypes.data, self.mats.size) == 0
        for i, t in enumerate(self.tex):
            assert L.refsh_set_texture(i, t.ctypes.data, t.shape[1], t.shape[0], t.shape[2] if t.ndim == 3 else 1) == 0

    def render(self, u, region=None, threads=0, out=None) -> np.ndarray:
        self.bind()
        u = np.ascontiguousarray(u, dtype=rt.UNIFORMS)
        w, h = int(u["width"][0]), int(u["height"][0])
        if out is None:
            out = np.zeros((h, w, 4), np.float32)
        x0, y0, x1, y1 = region if region is not None else (0, 0, w, h)
        assert self.L.refsh_render_region(u.ctypes.data, out.ctypes.data, x0, y0, x1, y1, threads) == 0
        return out


def render(scene, u, spec_math=True, threads=0) -> np.ndarray:
    """One dispatch of the reference shader over the whole image → RGBA32F, row 0 = bottom."""
    return Loaded(scene, spec_math).render(u, threads=threads)
