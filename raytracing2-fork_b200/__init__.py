"""raytracing2-fork_b200 — B200-native path-tracing backend for jackbaggins/RayTracing2-fork.

This package is a thin ctypes view of two in-tree native libraries (built by ``make`` in this
directory or by ``__graft_entry__.build()``):

* ``librt_b200.so`` — the CUDA backend behind the C-ABI of ``include/rt_b200.h`` (hand-written
  sm_100a kernels: BVH build, wavefront raygen / extend / shade, resolve, finalize).  There is no CPU
  fallback: :class:`Backend` raises if the library or a CUDA device is missing.
* ``librt_host.so`` — host-side scene assembly with the reference's surface (containers, camera,
  fixed materials, synthetic meshes, PNG out; ``host/rt_host.h``).

The package name contains a hyphen, so import it with
``importlib.import_module("raytracing2-fork_b200")``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(_HERE)

# ------------------------------------------------------------------------------------------------
# wire structs (include/rt_b200.h) as numpy dtypes — byte-for-byte the reference's structs
TRIANGLE = np.dtype(
    [("a", "<f4", 4), ("b", "<f4", 4), ("c", "<f4", 4), ("aTex", "<f4", 2), ("bTex", "<f4", 2),
     ("cTex", "<f4", 2), ("materialIndex", "<i4"), ("pad", "<f4")]
)
MATERIAL = np.dtype(
    [("color", "<f4", 4), ("specularColor", "<f4", 4), ("emissionColor", "<f4", 4),
     ("textureIndex", "<i4"), ("emissionStrength", "<f4"), ("smoothness", "<f4"),
     ("specularProbability", "<f4"), ("checkerScale", "<f4"), ("refractiveIndex", "<f4"),
     ("materialType", "<i4"), ("index", "<i4"), ("isEdgeHighlight", "<i4"), ("pad1", "<i4"),
     ("pad2", "<i4"), ("pad3", "<i4")]
)
UNIFORMS = np.dtype(
    [("pad", "<i4"), ("numTextures", "<i4"), ("width", "<u4"), ("height", "<u4"),
     ("numSpheres", "<i4"), ("numTriangles", "<i4"), ("basicShading", "<i4"),
     ("basicShadingShadow", "<i4"), ("basicShadingLightPosition", "<f4", 4),
     ("environmentalLight", "<i4"), ("maxBounceCount", "<i4"), ("numRaysPerPixel", "<i4"),
     ("frameIndex", "<u4"), ("cameraPos", "<f4", 4), ("viewportRight", "<f4", 4),
     ("viewportUp", "<f4", 4), ("viewportFront", "<f4", 4), ("pixelRight", "<f4", 4),
     ("pixelUp", "<f4", 4), ("defocusDiskRight", "<f4", 4), ("defocusDiskUp", "<f4", 4)]
)
REF_NODE = np.dtype(
    [("bmin", "<f4", 3), ("pad0", "<f4"), ("bmax", "<f4", 3), ("pad1", "<f4"),
     ("triangleIndex", "<i4"), ("triangleCount", "<i4"), ("childIndex", "<i4"), ("pad2", "<i4")]
)
BVH_NODE = np.dtype(
    [("lo_x", "<f4", 2), ("hi_x", "<f4", 2), ("lo_y", "<f4", 2), ("hi_y", "<f4", 2),
     ("lo_z", "<f4", 2), ("hi_z", "<f4", 2), ("child", "<i4", 2), ("count", "<i4", 2)]
)
assert TRIANGLE.itemsize == 80 and MATERIAL.itemsize == 96 and UNIFORMS.itemsize == 192
assert REF_NODE.itemsize == 48 and BVH_NODE.itemsize == 64

MAT_DIFFUSE, MAT_SPECULAR, MAT_LIGHT, MAT_CHECKER, MAT_GLASS, MAT_TEXTURE, MAT_GLASS_HIGHLIGHT = range(7)
RNG_REF_PCG, RNG_PHILOX = 0, 1
SPLIT_NONE, SPLIT_TILES, SPLIT_FRAMES = 0, 1, 2
FIRST_HIT_CENTRE, FIRST_HIT_SAMPLE0 = 0, 1


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("rng_mode", C.c_int32), ("split_mode", C.c_int32),
                ("rank", C.c_int32), ("world_size", C.c_int32), ("band_rows", C.c_int32),
                ("instrument", C.c_int32), ("kernel_timing", C.c_int32),
                ("max_paths_in_flight", C.c_uint64)]


class Counters(C.Structure):
    _fields_ = [("segments", C.c_uint64), ("paths", C.c_uint64), ("node_visits", C.c_uint64),
                ("tri_tests", C.c_uint64), ("extend_launches", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("extend_ms", C.c_double), ("shade_ms", C.c_double),
                ("build_ms", C.c_double), ("bvh_nodes", C.c_uint64), ("bvh_bytes", C.c_uint64),
                ("bvh_depth", C.c_uint64), ("bvh_width", C.c_uint64), ("bvh_stack_need", C.c_uint64),
                ("bvh_build_rounds", C.c_uint64), ("extend_blocks_per_sm", C.c_uint64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class Camera(C.Structure):
    """rth_camera — the reference's Camera state (camera.h:38-86)."""
    _fields_ = [("scrWidth", C.c_float), ("scrHeight", C.c_float), ("aspectRatio", C.c_float),
                ("mouseSensitivity", C.c_float), ("position", C.c_float * 3), ("right", C.c_float * 3),
                ("up", C.c_float * 3), ("front", C.c_float * 3), ("worldUp", C.c_float * 3),
                ("pitch", C.c_float), ("yaw", C.c_float), ("speed", C.c_float),
                ("lastX", C.c_double), ("lastY", C.c_double), ("firstMouse", C.c_int32),
                ("zoomSensitivity", C.c_float), ("zoom", C.c_float), ("hfov", C.c_float),
                ("viewportRight", C.c_float * 3), ("viewportUp", C.c_float * 3),
                ("viewportFront", C.c_float * 3), ("pixelRight", C.c_float * 3),
                ("pixelUp", C.c_float * 3), ("focusDistance", C.c_float),
                ("defocusAngle", C.c_float), ("defocusSensitivity", C.c_float),
                ("defocusDiskRight", C.c_float * 3), ("defocusDiskUp", C.c_float * 3)]


class Defaults(C.Structure):
    _fields_ = [("scr_width", C.c_int32), ("scr_height", C.c_int32), ("max_bounce_count", C.c_int32),
                ("num_rays_per_pixel", C.c_float), ("rays_per_pixel_sensitivity", C.c_float),
                ("basic_shading", C.c_int32), ("basic_shading_shadow", C.c_int32),
                ("basic_shading_environmental_light", C.c_int32), ("light_position", C.c_float * 3),
                ("screenshot_basic_shading", C.c_int32), ("screenshot_environmental_light", C.c_int32),
                ("screenshot_max_bounce_count", C.c_int32), ("screenshot_rays_per_pixel", C.c_int32),
                ("screenshot_frames", C.c_int32), ("cornell_light_brightness", C.c_float),
                ("cornell_padding", C.c_float), ("cornell_light_size", C.c_float),
                ("max_speed", C.c_float), ("hfov", C.c_float), ("pitch", C.c_float), ("yaw", C.c_float),
                ("focus_distance", C.c_float), ("defocus_angle", C.c_float), ("zoom", C.c_float),
                ("camera_pos", C.c_float * 3)]


class BackendError(RuntimeError):
    pass


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f3(v: Sequence[float]):
    return (C.c_float * 3)(*[float(x) for x in v])


# ------------------------------------------------------------------------------------------------
_host_lib = None
_backend_lib = None


def host_lib() -> C.CDLL:
    """librt_host.so (pure C++)."""
    global _host_lib
    if _host_lib is None:
        path = os.path.join(_HERE, "librt_host.so")
        if not os.path.exists(path):
            raise BackendError(f"{path} missing — run `make -C {_HERE}` or __graft_entry__.build()")
        L = C.CDLL(path)
        L.rth_scene_create.restype = C.c_void_p
        L.rth_last_error.restype = C.c_char_p
        L.rth_scene_triangle_count.restype = C.c_int64
        L.rth_scene_triangles.restype = C.c_void_p
        L.rth_scene_materials.restype = C.c_void_p
        L.rth_scene_texture.restype = C.c_void_p
        L.rth_adjust_rays_per_pixel.restype = C.c_float
        for name in ("rth_scene_destroy", "rth_scene_triangle_count", "rth_scene_triangles",
                     "rth_scene_material_count", "rth_scene_materials", "rth_scene_texture_count"):
            getattr(L, name).argtypes = [C.c_void_p]
        _host_lib = L
    return _host_lib


def backend_lib() -> C.CDLL:
    """librt_b200.so (CUDA, sm_100a).  Raises if it has not been built: no fallback exists."""
    global _backend_lib
    if _backend_lib is None:
        # RT_B200_LIB: another build of the SAME C-ABI (used only to A/B older kernel versions)
        path = os.environ.get("RT_B200_LIB") or os.path.join(_HERE, "librt_b200.so")
        if not os.path.exists(path):
            raise BackendError(f"{path} missing — the CUDA backend is required (no CPU fallback); "
                               f"run `make -C {_HERE}` or __graft_entry__.build()")
        L = C.CDLL(path)
        L.rt_last_error.restype = C.c_char_p
        L.rt_last_error.argtypes = [C.c_void_p]
        L.rt_version.restype = C.c_char_p
        L.rt_split_rows.restype = C.c_int64
        L.rt_split_frames.restype = C.c_int64
        _backend_lib = L
    return _backend_lib


# the symbols include/rt_b200.h declares; tests check that the library exports every one
ABI_SYMBOLS = [
    "rt_create", "rt_destroy", "rt_last_error", "rt_version", "rt_set_stream",
    "rt_scene_set_triangles", "rt_scene_set_materials", "rt_scene_set_texture", "rt_scene_build",
    "rt_render_frame", "rt_read_frame_rgba32f", "rt_screenshot", "rt_screenshot_device",
    "rt_screenshot_fetch", "rt_screenshot_partial", "rt_read_frame_sum", "rt_finalize_sums", "rt_first_hit", "rt_trace_rays",
    "rt_query_closest", "rt_query_occluded", "rt_query_nearest", "rt_scene_get_bvh", "rt_get_counters",
    "rt_reset_counters", "rt_comm_unique_id", "rt_comm_init", "rt_split_rows", "rt_split_frames", "rt_plan_batches",
]


# ------------------------------------------------------------------------------------------------
class Scene:
    """Host-side scene (rth_scene): triangles + materials + <=5 textures, reference containers."""

    def __init__(self):
        self.L = host_lib()
        self.h = C.c_void_p(self.L.rth_scene_create())

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.L.rth_scene_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def _chk(self, rc):
        if rc != 0:
            raise BackendError(f"host error {rc}: {self.L.rth_last_error().decode()}")

    # materials (mesh.h:49-102; rayTracing.cpp:1268-1283)
    def add_fixed_materials(self) -> int:
        return self.L.rth_add_fixed_materials(self.h)

    def add_diffuse(self, r, g, b) -> int:
        return self.L.rth_add_diffuse(self.h, C.c_float(r), C.c_float(g), C.c_float(b))

    def add_light(self, r, g, b, strength) -> int:
        return self.L.rth_add_light(self.h, C.c_float(r), C.c_float(g), C.c_float(b), C.c_float(strength))

    def add_specular(self, col, spec, smoothness, prob) -> int:
        return self.L.rth_add_specular(self.h, *[C.c_float(x) for x in (*col, *spec, smoothness, prob)])

    def add_checker(self, scale) -> int:
        return self.L.rth_add_checker(self.h, C.c_float(scale))

    def add_glass(self, col, ri) -> int:
        return self.L.rth_add_glass(self.h, *[C.c_float(x) for x in (*col, ri)])

    def add_textured(self, tex_index) -> int:
        return self.L.rth_add_textured(self.h, C.c_int32(tex_index))

    def add_material(self, m: np.ndarray) -> int:
        m = np.ascontiguousarray(m, dtype=MATERIAL).reshape(1)
        return self.L.rth_add_material(self.h, _ptr(m))

    # geometry (rayTracing.cpp:388-1118)
    def add_triangles(self, tris: np.ndarray):
        tris = np.ascontiguousarray(tris, dtype=TRIANGLE)
        self._chk(self.L.rth_add_triangles(self.h, _ptr(tris), C.c_int64(tris.size)))

    def add_cube(self, center, size, rotation, material):
        self._chk(self.L.rth_add_cube(self.h, _f3(center), _f3(size), _f3(rotation), C.c_int32(material)))

    def create_classic_cornell_box(self, room_size, red, green, white, light):
        self._chk(self.L.rth_create_classic_cornell_box(self.h, C.c_float(room_size), red, green, white, light))

    def create_diverse_cornell_box(self, room_size, red, green, white, light, glass, mirror, checker, metal):
        self._chk(self.L.rth_create_diverse_cornell_box(self.h, C.c_float(room_size), red, green, white,
                                                       light, glass, mirror, checker, metal))

    def add_cornell_box(self, light_size, pad, light, light_enabled=True):
        self._chk(self.L.rth_add_cornell_box(self.h, C.c_float(light_size), C.c_float(pad), light,
                                             int(light_enabled)))

    def add_mirror_cornell_box(self, light_size, pad, light, mirror):
        self._chk(self.L.rth_add_mirror_cornell_box(self.h, C.c_float(light_size), C.c_float(pad), light, mirror))

    def add_side_lit_cornell_box(self, light_size, pad, light, wall, rotate=False):
        self._chk(self.L.rth_add_side_lit_cornell_box(self.h, C.c_float(light_size), C.c_float(pad), light,
                                                      wall, int(rotate)))

    def add_sky_light_plane(self, light):
        self._chk(self.L.rth_add_sky_light_plane(self.h, light))

    def add_displaced_sphere(self, n, center, radius, amp, material):
        self._chk(self.L.rth_add_displaced_sphere(self.h, C.c_int32(n), _f3(center), C.c_float(radius),
                                                  C.c_float(amp), C.c_int32(material)))

    def set_procedural_texture(self, slot, size):
        self._chk(self.L.rth_set_procedural_texture(self.h, slot, size))

    def set_texture(self, slot, pixels: np.ndarray):
        px = np.ascontiguousarray(pixels, dtype=np.uint8)
        h, w = px.shape[0], px.shape[1]
        ch = 1 if px.ndim == 2 else px.shape[2]
        self._chk(self.L.rth_set_texture(self.h, slot, _ptr(px), w, h, ch))

    def load_model_folder(self, folder: str):
        """getTrianglesData_(folder, ...) of mesh.h:279 on a fresh scene (OBJ + MTL + textures/*.png)."""
        self._chk(self.L.rth_load_model_folder(self.h, folder.encode()))

    def save(self, path):
        self._chk(self.L.rth_scene_save(self.h, path.encode()))

    def load(self, path):
        self._chk(self.L.rth_scene_load(self.h, path.encode()))

    # views
    @property
    def triangles(self) -> np.ndarray:
        n = self.L.rth_scene_triangle_count(self.h)
        if n == 0:
            return np.zeros(0, dtype=TRIANGLE)
        buf = (C.c_char * (n * 80)).from_address(self.L.rth_scene_triangles(self.h))
        return np.frombuffer(buf, dtype=TRIANGLE).copy()

    @property
    def materials(self) -> np.ndarray:
        n = self.L.rth_scene_material_count(self.h)
        buf = (C.c_char * (n * 96)).from_address(self.L.rth_scene_materials(self.h))
        return np.frombuffer(buf, dtype=MATERIAL).copy()

    @property
    def textures(self):
        out = []
        for i in range(self.L.rth_scene_texture_count(self.h)):
            w, h, ch = C.c_int32(), C.c_int32(), C.c_int32()
            p = self.L.rth_scene_texture(self.h, i, C.byref(w), C.byref(h), C.byref(ch))
            buf = (C.c_char * (w.value * h.value * ch.value)).from_address(p)
            out.append(np.frombuffer(buf, dtype=np.uint8).reshape(h.value, w.value, ch.value).copy())
        return out


def defaults() -> Defaults:
    d = Defaults()
    host_lib().rth_get_defaults(C.byref(d))
    return d


def make_camera(width, height, pos, hfov=None, pitch=None, yaw=None, focus=None, defocus=None,
                zoom=None, speed=None) -> Camera:
    """Camera(...) of camera.h:99 with the reference's start values (rayTracing.cpp:82-89) as defaults."""
    d = defaults()
    c = Camera()
    host_lib().rth_camera_init(
        C.byref(c), int(width), int(height), C.c_float(d.max_speed if speed is None else speed), _f3(pos),
        C.c_float(d.hfov if hfov is None else hfov), C.c_float(d.pitch if pitch is None else pitch),
        C.c_float(d.yaw if yaw is None else yaw), C.c_float(d.focus_distance if focus is None else focus),
        C.c_float(d.defocus_angle if defocus is None else defocus), C.c_float(d.zoom if zoom is None else zoom))
    return c


def screenshot_uniforms(scene: Scene, cam: Camera, *, spp=None, max_bounce=None, env_light=None,
                        frame_index=0) -> np.ndarray:
    """The uniform block screenshot() uses (rayTracing.cpp:146-150), optionally overridden."""
    u = np.zeros(1, dtype=UNIFORMS)
    host_lib().rth_fill_screenshot_uniforms(scene.h, C.byref(cam), _ptr(u))
    if spp is not None:
        u["numRaysPerPixel"] = spp
    if max_bounce is not None:
        u["maxBounceCount"] = max_bounce
    if env_light is not None:
        u["environmentalLight"] = int(env_light)
    u["frameIndex"] = frame_index
    return u


def interactive_uniforms(scene: Scene, cam: Camera, rays_per_pixel=5.0, frame_index=0) -> np.ndarray:
    u = np.zeros(1, dtype=UNIFORMS)
    host_lib().rth_fill_interactive_uniforms(scene.h, C.byref(cam), C.c_float(rays_per_pixel),
                                             C.c_uint32(frame_index), _ptr(u))
    return u


def write_png(path: str, rgb8: np.ndarray):
    px = np.ascontiguousarray(rgb8, dtype=np.uint8)
    h, w = px.shape[0], px.shape[1]
    ch = 1 if px.ndim == 2 else px.shape[2]
    rc = host_lib().rth_write_png(path.encode(), w, h, ch, _ptr(px))
    if rc:
        raise BackendError(host_lib().rth_last_error().decode())


# ------------------------------------------------------------------------------------------------
class Backend:
    """One rt_ctx = one GPU.  Mirrors the reference's upload / dispatch / readback call sequence
    (rayTracing.cpp:1293, :1323-1325, :1402-1406, :124-283) through the C-ABI."""

    def __init__(self, device=0, rng_mode=RNG_PHILOX, split_mode=SPLIT_NONE, rank=0, world_size=1,
                 band_rows=0, instrument=False, kernel_timing=False, max_paths_in_flight=0):
        self.L = backend_lib()
        cfg = Config(device, rng_mode, split_mode, rank, world_size, band_rows, int(instrument),
                     int(kernel_timing),
                     max_paths_in_flight)
        self.cfg = cfg
        self.h = C.c_void_p()
        rc = self.L.rt_create(C.byref(self.h), C.byref(cfg))
        if rc != 0:
            msg = self.L.rt_last_error(self.h).decode() if self.h else self.L.rt_last_error(None).decode()
            self.h = None
            raise BackendError(f"rt_create failed ({rc}): {msg}")
        self.width = self.height = 0
        self._stream_ptr = 0       # the stream the ctx is bound to (0 = the ctx's own stream, unknown to torch)
        self._query_stream = None  # its torch view, made by the first ray query

    def close(self):
        if getattr(self, "h", None):
            self.L.rt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != 0:
            raise BackendError(f"rt error {rc}: {self.L.rt_last_error(self.h).decode()}")

    def set_stream(self, cuda_stream_ptr: int):
        self._chk(self.L.rt_set_stream(self.h, C.c_void_p(cuda_stream_ptr)))
        self._stream_ptr = int(cuda_stream_ptr or 0)
        self._query_stream = None

    def set_triangles(self, tris: np.ndarray):
        tris = np.ascontiguousarray(tris, dtype=TRIANGLE)
        self._chk(self.L.rt_scene_set_triangles(self.h, _ptr(tris), C.c_int64(tris.size)))

    def set_materials(self, mats: np.ndarray):
        mats = np.ascontiguousarray(mats, dtype=MATERIAL)
        self._chk(self.L.rt_scene_set_materials(self.h, _ptr(mats), C.c_int32(mats.size)))

    def set_texture(self, slot: int, pixels: np.ndarray):
        px = np.ascontiguousarray(pixels, dtype=np.uint8)
        h, w = px.shape[0], px.shape[1]
        ch = 1 if px.ndim == 2 else px.shape[2]
        self._chk(self.L.rt_scene_set_texture(self.h, slot, _ptr(px), w, h, ch))

    def build(self):
        self._chk(self.L.rt_scene_build(self.h))

    def upload(self, scene: Scene):
        """set_triangles + set_materials + set_texture* + build, straight from a host Scene."""
        self.set_triangles(scene.triangles)
        self.set_materials(scene.materials)
        for i, t in enumerate(scene.textures):
            self.set_texture(i, t)
        self.build()

    def render_frame(self, u: np.ndarray):
        u = np.ascontiguousarray(u, dtype=UNIFORMS)
        self.width, self.height = int(u["width"][0]), int(u["height"][0])
        self._chk(self.L.rt_render_frame(self.h, _ptr(u)))

    def read_frame(self) -> np.ndarray:
        out = np.zeros((self.height, self.width, 4), dtype=np.float32)
        self._chk(self.L.rt_read_frame_rgba32f(self.h, _ptr(out)))
        return out

    def screenshot(self, u: np.ndarray, frames: int, want_output=True) -> Optional[np.ndarray]:
        u = np.ascontiguousarray(u, dtype=UNIFORMS)
        self.width, self.height = int(u["width"][0]), int(u["height"][0])
        out = np.zeros((self.height, self.width, 3), dtype=np.uint8) if want_output else None
        self._chk(self.L.rt_screenshot(self.h, _ptr(u), C.c_int32(frames), _ptr(out)))
        return out

    def screenshot_device(self, u: np.ndarray, frames: int):
        u = np.ascontiguousarray(u, dtype=UNIFORMS)
        self.width, self.height = int(u["width"][0]), int(u["height"][0])
        self._chk(self.L.rt_screenshot_device(self.h, _ptr(u), C.c_int32(frames)))

    def screenshot_fetch(self) -> np.ndarray:
        out = np.zeros((self.height, self.width, 3), dtype=np.uint8)
        self._chk(self.L.rt_screenshot_fetch(self.h, _ptr(out)))
        return out

    def screenshot_partial(self, u: np.ndarray, frames: int) -> np.ndarray:
        """This rank's share of a screenshot: the 8-bit frame sums (H, W, 3) u32, row 0 = bottom."""
        u = np.ascontiguousarray(u, dtype=UNIFORMS)
        self.width, self.height = int(u["width"][0]), int(u["height"][0])
        self._chk(self.L.rt_screenshot_partial(self.h, _ptr(u), C.c_int32(frames)))
        sums = np.zeros((self.height, self.width, 3), dtype=np.uint32)
        self._chk(self.L.rt_read_frame_sum(self.h, _ptr(sums)))
        return sums

    def finalize_sums(self, sums: np.ndarray, frames: int) -> np.ndarray:
        sums = np.ascontiguousarray(sums, dtype=np.uint32)
        h, w = sums.shape[:2]
        out = np.zeros((h, w, 3), dtype=np.uint8)
        self._chk(self.L.rt_finalize_sums(self.h, _ptr(sums), w, h, C.c_int32(frames), _ptr(out)))
        return out

    def first_hit(self, u: np.ndarray, mode=FIRST_HIT_CENTRE):
        u = np.ascontiguousarray(u, dtype=UNIFORMS)
        w, h = int(u["width"][0]), int(u["height"][0])
        tri = np.zeros((h, w), dtype=np.int32)
        dst = np.zeros((h, w), dtype=np.float32)
        self._chk(self.L.rt_first_hit(self.h, _ptr(u), C.c_int32(mode), _ptr(tri), _ptr(dst)))
        return tri, dst

    def trace_rays(self, origins: np.ndarray, dirs: np.ndarray):
        o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, 3)
        n = o.shape[0]
        tri = np.zeros(n, dtype=np.int32)
        dst = np.zeros(n, dtype=np.float32)
        bu = np.zeros(n, dtype=np.float32)
        bv = np.zeros(n, dtype=np.float32)
        self._chk(self.L.rt_trace_rays(self.h, _ptr(o), _ptr(d), C.c_int64(n), _ptr(tri), _ptr(dst),
                                       _ptr(bu), _ptr(bv)))
        return tri, dst, bu, bv

    # ---- queries on CUDA tensors (rt_query_closest / rt_query_occluded / rt_query_nearest)
    def _stream_for_queries(self, torch):
        """The torch view of the stream the ctx launches on.  The ctx is bound once: to the stream given to
        set_stream, or else to a private stream made here (rt_set_stream synchronises the previous stream, so it is
        never called per query)."""
        if self._query_stream is None:
            dev = torch.device("cuda", self.cfg.device)
            if self._stream_ptr:
                self._query_stream = torch.cuda.ExternalStream(self._stream_ptr, device=dev)
            else:
                s = torch.cuda.Stream(device=dev)
                self.set_stream(s.cuda_stream)
                self._query_stream = s
        return self._query_stream

    def _query_inputs(self, torch, inputs, bound, bound_name):
        """inputs: (name, tensor) pairs, each a float32 (N, 3) CUDA tensor, the first defining N; bound (tmax or
        max_dist): None, a float or a float32 (N,) CUDA tensor.  Returns N, the contiguous inputs and the bound."""
        dev = torch.device("cuda", self.cfg.device)

        def check(t, what, shape):
            if not isinstance(t, torch.Tensor):
                raise BackendError(f"{what} must be a torch tensor")
            if t.device != dev:
                raise BackendError(f"{what} is on {t.device}, the backend's device is {dev}")
            if t.dtype != torch.float32:
                raise BackendError(f"{what} must be float32, not {t.dtype}")
            if tuple(t.shape) != shape:
                raise BackendError(f"{what} has shape {tuple(t.shape)}, expected {shape}")
            return t.contiguous()

        first_name, first = inputs[0]
        n = first.shape[0] if isinstance(first, torch.Tensor) and first.dim() == 2 else -1
        if n < 0:
            raise BackendError(f"{first_name} must be a float32 (N, 3) CUDA tensor")
        arrays = [check(t, name, (n, 3)) for name, t in inputs]
        if bound is None:
            b = None
        elif isinstance(bound, (int, float)) and not isinstance(bound, bool):
            b = torch.full((n,), float(bound), dtype=torch.float32, device=dev)
        else:
            b = check(bound, bound_name, (n,))
        return n, arrays, b

    def _run_query(self, torch, fn, tensors, args):
        """Enqueue one query ordered after the current torch stream's work and before whatever it does next, with no
        host synchronisation: the query stream waits for the current stream, the current stream waits for the query."""
        cur = torch.cuda.current_stream(torch.device("cuda", self.cfg.device))
        qs = self._stream_for_queries(torch)
        qs.wait_stream(cur)
        self._chk(fn(self.h, *args))
        cur.wait_stream(qs)
        for t in tensors:   # the caching allocator must not hand these out again before the query has run
            if t is not None:
                t.record_stream(qs)

    @staticmethod
    def _dptr(t):
        return C.c_void_p(None if t is None else t.data_ptr())

    def query_closest(self, origins, dirs, tmax=None):
        """Closest hit of every ray on the device: origins / dirs float32 (N, 3) CUDA tensors; tmax None (unbounded),
        a float or a float32 (N,) tensor.  Returns (tri_id int32, dst, u, v), (N,) tensors: the result of trace_rays
        for the same ray when its distance is below tmax, else the miss -1 / 1e38 / 0 / 0."""
        import torch
        n, (o, d), tm = self._query_inputs(torch, (("origins", origins), ("dirs", dirs)), tmax, "tmax")
        dev = o.device
        tri = torch.empty(n, dtype=torch.int32, device=dev)
        dst, bu, bv = (torch.empty(n, dtype=torch.float32, device=dev) for _ in range(3))
        self._run_query(torch, self.L.rt_query_closest, (o, d, tm, tri, dst, bu, bv),
                        (self._dptr(o), self._dptr(d), self._dptr(tm), C.c_int64(n), self._dptr(tri),
                         self._dptr(dst), self._dptr(bu), self._dptr(bv)))
        return tri, dst, bu, bv

    def query_occluded(self, origins, dirs, tmax=None):
        """Is anything hit with t < tmax?  Same inputs as query_closest; returns a bool (N,) CUDA tensor.  The walk
        stops at the first triangle it accepts."""
        import torch
        n, (o, d), tm = self._query_inputs(torch, (("origins", origins), ("dirs", dirs)), tmax, "tmax")
        occ = torch.empty(n, dtype=torch.bool, device=o.device)   # one byte per element, written as 0 / 1
        self._run_query(torch, self.L.rt_query_occluded, (o, d, tm, occ),
                        (self._dptr(o), self._dptr(d), self._dptr(tm), C.c_int64(n), self._dptr(occ)))
        return occ

    def query_nearest(self, points, max_dist=None):
        """Nearest triangle of every point on the device: points a float32 (N, 3) CUDA tensor; max_dist None
        (unbounded), a float or a float32 (N,) tensor.  Returns (tri_id int32, dist, u, v, closest (N, 3)): among the
        triangles closer than max_dist (and 1e38), the nearest one, exact ties to the lowest id, with the barycentrics
        of the closest point a + (b - a) u + (c - a) v and that point; a miss is -1 / 1e38 / 0 / 0 / (0, 0, 0).  A NaN,
        zero or negative max_dist and a non-finite point miss.  Ordered on the current stream like query_closest."""
        import torch
        n, (p,), md = self._query_inputs(torch, (("points", points),), max_dist, "max_dist")
        dev = p.device
        tri = torch.empty(n, dtype=torch.int32, device=dev)
        dist, bu, bv = (torch.empty(n, dtype=torch.float32, device=dev) for _ in range(3))
        closest = torch.empty((n, 3), dtype=torch.float32, device=dev)
        self._run_query(torch, self.L.rt_query_nearest, (p, md, tri, dist, bu, bv, closest),
                        (self._dptr(p), self._dptr(md), C.c_int64(n), self._dptr(tri), self._dptr(dist),
                         self._dptr(bu), self._dptr(bv), self._dptr(closest)))
        return tri, dist, bu, bv, closest

    def get_bvh(self):
        nn, nt = C.c_int64(), C.c_int64()
        lo, hi = (C.c_float * 3)(), (C.c_float * 3)()
        self._chk(self.L.rt_scene_get_bvh(self.h, None, C.byref(nn), None, C.byref(nt), lo, hi))
        nodes = np.zeros(max(nn.value, 1), dtype=BVH_NODE)
        ids = np.zeros(max(nt.value, 1), dtype=np.int32)
        self._chk(self.L.rt_scene_get_bvh(self.h, _ptr(nodes), C.byref(nn), _ptr(ids), C.byref(nt), lo, hi))
        return nodes[: nn.value], ids[: nt.value], np.array(lo[:]), np.array(hi[:])

    def counters(self) -> dict:
        c = Counters()
        self._chk(self.L.rt_get_counters(self.h, C.byref(c)))
        return c.as_dict()

    def reset_counters(self):
        self._chk(self.L.rt_reset_counters(self.h))

    # multi-GPU plumbing: the 128-byte NCCL id travels through whatever the host has
    def comm_unique_id(self) -> bytes:
        buf = (C.c_uint8 * 128)()
        self._chk(self.L.rt_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, uid: bytes):
        buf = (C.c_uint8 * 128).from_buffer_copy(uid)
        self._chk(self.L.rt_comm_init(self.h, buf))


def split_rows(height, band_rows, rank, world) -> np.ndarray:
    out = np.zeros(height, dtype=np.int32)
    n = backend_lib().rt_split_rows(C.c_int32(height), C.c_int32(band_rows), C.c_int32(rank),
                                    C.c_int32(world), _ptr(out), C.c_int64(height))
    return out[:n]


def plan_batches(max_paths_in_flight, local_pixels, spp, frames, rng_mode=1):
    """(samples of a frame per batch, frames per batch) rt_screenshot will use — host arithmetic only."""
    s, f = C.c_int32(0), C.c_int32(0)
    rc = backend_lib().rt_plan_batches(C.c_uint64(max_paths_in_flight), C.c_int64(local_pixels), C.c_int32(spp),
                                       C.c_int32(frames), C.c_int32(rng_mode), C.byref(s), C.byref(f))
    if rc:
        raise BackendError(f"rt_plan_batches failed ({rc})")
    return s.value, f.value


def split_frames(frames, rank, world) -> np.ndarray:
    out = np.zeros(max(frames, 1), dtype=np.int32)
    n = backend_lib().rt_split_frames(C.c_int32(frames), C.c_int32(rank), C.c_int32(world), _ptr(out),
                                      C.c_int64(frames))
    return out[:n]


# ------------------------------------------------------------------------------------------------
# named scenes of BASELINE.md §3 (host-side assembly only; no GPU needed)
def scene_classic_cornell() -> Scene:
    """Config 1: createClassicCornellBox(10, ...) with no OBJ: 38 triangles, 6 materials."""
    s = Scene()
    red = s.add_fixed_materials()
    s.create_classic_cornell_box(10.0, red, red + 1, red + 2, red + 3)
    return s


def scene_textured_sphere(n_quads=224, container="cornell", tex_size=1024) -> Scene:
    """Configs 2/3/5: synthetic textured displaced sphere (2·n² triangles) inside addCornellBox /
    addMirrorCornellBox with the reference constants (0.17, 0.3, light 15.0)."""
    d = defaults()
    s = Scene()
    s.set_procedural_texture(0, tex_size)
    mat = s.add_textured(0)
    s.add_displaced_sphere(n_quads, (0.0, 0.0, 0.0), 3.0, 0.05, mat)
    red = s.add_fixed_materials()
    if container == "cornell":
        s.add_cornell_box(d.cornell_light_size, d.cornell_padding, red + 3, True)
    elif container == "mirror":
        s.add_mirror_cornell_box(d.cornell_light_size, d.cornell_padding, red + 3, red + 4)
    elif container != "none":
        raise ValueError(container)
    return s


def scene_from_rtsc(path: str, container="cornell") -> Scene:
    """A model written by the reference's loader (tools/make_assets.sh → assets/_gen/<model>.rtsc: triangles,
    the material table INCLUDING the five fixed materials, decoded textures) inside a reference container —
    config 2(i)/3(i) with `Data/robot`."""
    d = defaults()
    s = Scene()
    s.load(path)
    n = s.materials.size
    if container == "cornell":
        s.add_cornell_box(d.cornell_light_size, d.cornell_padding, n - 2, True)
    elif container == "mirror":
        s.add_mirror_cornell_box(d.cornell_light_size, d.cornell_padding, n - 2, n - 1)
    elif container != "none":
        raise ValueError(container)
    return s


def scene_big_sphere(n_quads=2236) -> Scene:
    """Config 4: 2·n² ≈ 10 M-triangle diffuse displaced sphere in the classic Cornell room
    (walls + light, without the two cubes)."""
    s = Scene()
    red = s.add_fixed_materials()
    white = red + 2
    s.create_classic_cornell_box(10.0, red, red + 1, white, red + 3)
    tris = s.triangles[:14]  # 12 walls + 2 light triangles; drop the 24 cube triangles
    s2 = Scene()
    s2.add_fixed_materials()
    s2.add_triangles(tris)
    s2.add_displaced_sphere(n_quads, (0.0, -1.0, 0.0), 3.0, 0.05, white)
    return s2


def camera_for_box(scene: Scene, width, height, fill=0.98) -> Camera:
    """Camera on the +Z axis looking down -Z (yaw π/2) placed so that the scene's front face just
    fits the view — the role (0,0,15.5) plays for the classic box (BASELINE.md §3, config 1)."""
    t = scene.triangles
    pts = np.concatenate([t["a"][:, :3], t["b"][:, :3], t["c"][:, :3]])
    lo, hi = pts.min(0), pts.max(0)
    d = defaults()
    half_tan = 2 * np.tan(d.hfov / 2) / np.exp(d.zoom * 0.1)  # |viewportRight| / focus
    half_w = max((hi[0] - lo[0]) / 2, (hi[1] - lo[1]) / 2 * width / height)
    dist = half_w / (half_tan * fill)
    pos = ((lo[0] + hi[0]) / 2, (lo[1] + hi[1]) / 2, hi[2] + dist)
    return make_camera(width, height, pos)
