"""ctypes binding of the C ABI declared in include/shimmer_b200.h.

The binding is generic over the symbol prefix because the test oracle exposes the same
builder vocabulary under ``orc_``; the product only ever loads ``libshimmer_b200.so``
(prefix ``shim_``).  There is no fallback: if the CUDA library is missing, importing a
scene raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "lib" / "libshimmer_b200.so"


class ShimError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"[{code}] {message}")
        self.code = code
        self.message = message


class Camera(C.Structure):
    """The nine ``Camera::new`` arguments (reference src/camera.rs:44-54)."""

    _fields_ = [
        ("look_from", C.c_float * 3), ("look_at", C.c_float * 3), ("view_up", C.c_float * 3),
        ("vertical_fov", C.c_float), ("aspect_ratio", C.c_float), ("aperture", C.c_float),
        ("focus_dist", C.c_float), ("time_start", C.c_float), ("time_end", C.c_float),
    ]

    @classmethod
    def new(cls, look_from, look_at, view_up, vertical_fov, aspect_ratio, aperture, focus_dist,
            time_start=0.0, time_end=0.0) -> "Camera":
        c = cls()
        c.look_from[:] = [float(v) for v in look_from]
        c.look_at[:] = [float(v) for v in look_at]
        c.view_up[:] = [float(v) for v in view_up]
        c.vertical_fov = vertical_fov
        c.aspect_ratio = aspect_ratio
        c.aperture = aperture
        c.focus_dist = focus_dist
        c.time_start = time_start
        c.time_end = time_end
        return c

    def as_array15(self) -> np.ndarray:
        return np.array(list(self.look_from) + list(self.look_at) + list(self.view_up) +
                        [self.vertical_fov, self.aspect_ratio, self.aperture, self.focus_dist,
                         self.time_start, self.time_end], dtype=np.float32)


RENDER_RAW_SUM = 1
RENDER_PREDICTORS = 2
RENDER_COUNT_NODES = 4
RENDER_PROFILE = 8
RENDER_KEEP_PREDICTORS = 16
SHARD_SAMPLES = 0
SHARD_TILES = 1


class RenderParams(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("samples_per_pixel", C.c_int32), ("max_depth", C.c_int32),
        ("tile_width", C.c_int32), ("tile_height", C.c_int32), ("background", C.c_float * 3), ("seed", C.c_uint64),
        ("sample_begin", C.c_int32), ("sample_count", C.c_int32), ("tile_rank", C.c_int32), ("tile_world", C.c_int32),
        ("flags", C.c_int32), ("pool_paths", C.c_int32),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("rays", C.c_uint64), ("samples", C.c_uint64), ("node_visits", C.c_uint64), ("prim_tests", C.c_uint64),
        ("hrpp_true_positive", C.c_uint64), ("hrpp_false_positive", C.c_uint64), ("hrpp_no_prediction", C.c_uint64),
        ("kernel_launches", C.c_uint64), ("iterations", C.c_uint64), ("device_ms", C.c_double),
        ("extend_ms", C.c_double), ("shade_ms", C.c_double), ("generate_ms", C.c_double), ("extend_launches", C.c_uint64),
        ("extend_variant", C.c_uint64), ("pool_paths", C.c_uint64), ("pool_bytes", C.c_uint64), ("devices", C.c_uint64),
        ("wall_ms", C.c_double),
    ]

    EXTEND_KERNELS = {0: "wf_extend", 1: "wf_bvh1_walk", 2: "wf_extend_solo", 3: "wf_extend_list", 4: "wf_trace_solo"}

    def as_dict(self) -> dict:
        return {k: getattr(self, k) for k, _ in self._fields_}


class HitRecord(C.Structure):
    """``shim_hit_record``: the reference's ``HitRecord`` (hittable.rs:15-52) plus the id of what was hit (48 bytes)."""

    _fields_ = [
        ("point", C.c_float * 3), ("normal", C.c_float * 3), ("t", C.c_float), ("u", C.c_float), ("v", C.c_float),
        ("front_face", C.c_int32), ("material", C.c_int32), ("hittable", C.c_int32),
    ]


# the same record as a numpy structured dtype (same field offsets as HitRecord)
HIT_RECORD_DTYPE = np.dtype({
    "names": [n for n, _ in HitRecord._fields_],
    "formats": [(np.float32, (3,)), (np.float32, (3,)), np.float32, np.float32, np.float32, np.int32, np.int32, np.int32],
    "offsets": [getattr(HitRecord, n).offset for n, _ in HitRecord._fields_],
    "itemsize": C.sizeof(HitRecord),
})


_F, _I, _P = C.c_float, C.c_int, C.c_void_p
# builder vocabulary shared by the product (shim_) and the test oracle (orc_)
_BUILDER_SIGS = {
    "texture_solid": [_F, _F, _F],
    "texture_checker": [_F, _I, _I],
    "texture_marble": [_F, C.c_uint32],
    "texture_image": [C.c_void_p, _I, _I],
    "material_lambertian": [_I],
    "material_metal": [_F, _F, _F, _F],
    "material_dielectric": [_F],
    "material_diffuse_light": [_I],
    "material_isotropic": [_I],
    "sphere": [_F, _F, _F, _F, _I],
    "moving_sphere": [_F] * 9 + [_I],
    "xy_rect": [_F] * 5 + [_I],
    "xz_rect": [_F] * 5 + [_I],
    "yz_rect": [_F] * 5 + [_I],
    "tri": [C.c_void_p, _I],
    "cube": [_F] * 6 + [_I],
    "list_create": [],
    "list_add": [_I, _I],
    "tris_bulk": [C.c_void_p, _I, _I, _I],
    "bvh": [_I, _F, _F, C.c_uint64, _I],
    "translate": [_I, _F, _F, _F],
    "rotate_y": [_I, _F],
    "constant_medium": [_I, _F, _I],
    "world_add": [_I],
    "commit": [],
}


def bind_builder(lib: C.CDLL, prefix: str) -> None:
    getattr(lib, prefix + "scene_create").restype = _P
    getattr(lib, prefix + "scene_create").argtypes = []
    getattr(lib, prefix + "scene_destroy").restype = None
    getattr(lib, prefix + "scene_destroy").argtypes = [_P]
    getattr(lib, prefix + "last_error").restype = C.c_char_p
    getattr(lib, prefix + "last_error").argtypes = []
    for name, args in _BUILDER_SIGS.items():
        fn = getattr(lib, prefix + name)
        fn.restype = _I
        fn.argtypes = [_P] + args
    for name in ("bvh_info", "bvh_nodes"):
        fn = getattr(lib, prefix + name)
        fn.restype = _I
    if prefix == "shim_":
        lib.shim_scene_set_option.restype = _I
        lib.shim_scene_set_option.argtypes = [_P, _I, _I]
    getattr(lib, prefix + "bvh_info").argtypes = [_P, _I, _P, _P, _P]
    getattr(lib, prefix + "bvh_nodes").argtypes = [_P, _I, _P, _P, _P, _P]


_lib = None


def load_library() -> C.CDLL:
    """Loads libshimmer_b200.so (built in-tree by ``__graft_entry__.build()``); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("SHIMMER_B200_LIB", LIB_PATH))
    if not path.exists():
        raise ShimError(-3, f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(this backend has no CPU fallback)")
    lib = C.CDLL(str(path))
    bind_builder(lib, "shim_")
    lib.shim_version.restype = _I
    lib.shim_bvh_from_nodes.restype = _I
    lib.shim_bvh_from_nodes.argtypes = [_P, _I, _P, _P, _I, _F, _F, _I]
    lib.shim_scene_device_bytes.restype = C.c_uint64
    lib.shim_scene_device_bytes.argtypes = [_P]
    lib.shim_render.restype = _I
    lib.shim_render.argtypes = [_P, C.POINTER(Camera), C.POINTER(RenderParams), _P, C.POINTER(Stats)]
    lib.shim_render_device.restype = _I
    lib.shim_render_device.argtypes = [_P, C.POINTER(Camera), C.POINTER(RenderParams), _P, C.POINTER(Stats), _P]
    lib.shim_render_multi.restype = _I
    lib.shim_render_multi.argtypes = [_P, C.POINTER(Camera), C.POINTER(RenderParams), _I, _P, _I, _P, C.POINTER(Stats)]
    lib.shim_shutdown.restype = _I
    lib.shim_shutdown.argtypes = []
    lib.shim_pool_bytes.restype = C.c_uint64
    lib.shim_pool_bytes.argtypes = [_I]
    lib.shim_trace_closest.restype = _I
    lib.shim_trace_closest.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _P, _P, _P]
    lib.shim_trace_closest_device.restype = _I
    lib.shim_trace_closest_device.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _P, _P, _P]
    lib.shim_trace_hit.restype = _I
    lib.shim_trace_hit.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, C.POINTER(HitRecord), _P]
    lib.shim_trace_hit_device.restype = _I
    lib.shim_trace_hit_device.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, C.POINTER(HitRecord), _P]
    lib.shim_trace_occluded.restype = _I
    lib.shim_trace_occluded.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _P, _P]
    lib.shim_trace_occluded_device.restype = _I
    lib.shim_trace_occluded_device.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _P, _P]
    lib.shim_tile_layout.restype = _I
    lib.shim_tile_layout.argtypes = [_I, _I, _I, _I, _P, _I]
    lib.shim_camera_fields.restype = _I
    lib.shim_camera_fields.argtypes = [C.POINTER(Camera), _P]
    lib.shim_aabb_hit.restype = _I
    lib.shim_aabb_hit.argtypes = [_P, _P, _P, _P, _F, _F, _I]
    lib.shim_hrpp_hash.restype = C.c_uint64
    lib.shim_hrpp_hash.argtypes = [_P, _P]
    lib.shim_host_alloc.restype = _P
    lib.shim_host_alloc.argtypes = [C.c_size_t]
    lib.shim_host_free.restype = None
    lib.shim_host_free.argtypes = [_P]
    lib.shim_write_ppm.restype = C.c_int64
    lib.shim_write_ppm.argtypes = [_P, _I, _I, C.c_char_p]
    _lib = lib
    return lib


class SceneHandle:
    """Thin object wrapper over the builder calls of one library (``shim_`` or a test double)."""

    def __init__(self, lib: C.CDLL, prefix: str = "shim_"):
        self.lib = lib
        self.prefix = prefix
        self.ptr = getattr(lib, prefix + "scene_create")()
        if not self.ptr:
            raise ShimError(-1, "scene_create failed")
        self._keep = []

    def close(self):
        if getattr(self, "ptr", None):
            getattr(self.lib, self.prefix + "scene_destroy")(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _call(self, name, *args):
        rc = getattr(self.lib, self.prefix + name)(self.ptr, *args)
        if rc < 0:
            msg = getattr(self.lib, self.prefix + "last_error")()
            raise ShimError(rc, (msg or b"").decode())
        return rc

    # ---- textures
    def texture_solid(self, r, g, b): return self._call("texture_solid", r, g, b)
    def texture_checker(self, scale, even, odd): return self._call("texture_checker", scale, even, odd)
    def texture_marble(self, scale, seed): return self._call("texture_marble", scale, seed)

    def texture_image(self, rgb8: np.ndarray):
        a = np.ascontiguousarray(rgb8, dtype=np.uint8)
        assert a.ndim == 3 and a.shape[2] == 3
        return self._call("texture_image", a.ctypes.data, a.shape[1], a.shape[0])

    # ---- materials
    def material_lambertian(self, tex): return self._call("material_lambertian", tex)
    def material_metal(self, r, g, b, fuzz): return self._call("material_metal", r, g, b, fuzz)
    def material_dielectric(self, ior): return self._call("material_dielectric", ior)
    def material_diffuse_light(self, tex): return self._call("material_diffuse_light", tex)
    def material_isotropic(self, tex): return self._call("material_isotropic", tex)

    def lambertian_color(self, r, g, b): return self.material_lambertian(self.texture_solid(r, g, b))
    def diffuse_light_color(self, r, g, b): return self.material_diffuse_light(self.texture_solid(r, g, b))

    # ---- hittables
    def sphere(self, c, r, mat): return self._call("sphere", c[0], c[1], c[2], r, mat)

    def moving_sphere(self, c0, c1, t0, t1, r, mat):
        return self._call("moving_sphere", c0[0], c0[1], c0[2], c1[0], c1[1], c1[2], t0, t1, r, mat)

    def xy_rect(self, x0, x1, y0, y1, k, mat): return self._call("xy_rect", x0, x1, y0, y1, k, mat)
    def xz_rect(self, x0, x1, z0, z1, k, mat): return self._call("xz_rect", x0, x1, z0, z1, k, mat)
    def yz_rect(self, y0, y1, z0, z1, k, mat): return self._call("yz_rect", y0, y1, z0, z1, k, mat)

    def tri(self, p0, p1, p2, mat):
        a = np.array([*p0, *p1, *p2], dtype=np.float32)
        return self._call("tri", a.ctypes.data, mat)

    def cube(self, pmin, pmax, mat): return self._call("cube", pmin[0], pmin[1], pmin[2], pmax[0], pmax[1], pmax[2], mat)
    def list_create(self): return self._call("list_create")
    def list_add(self, lst, h): return self._call("list_add", lst, h)

    def tris_bulk(self, xyz: np.ndarray, mat, lst):
        a = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 9)
        return self._call("tris_bulk", a.ctypes.data, a.shape[0], mat, lst)

    def bvh(self, lst, t0=0.0, t1=1.0, seed=0, with_predictor=False):
        return self._call("bvh", lst, t0, t1, seed, 1 if with_predictor else 0)

    def translate(self, h, d): return self._call("translate", h, d[0], d[1], d[2])
    def rotate_y(self, h, deg): return self._call("rotate_y", h, deg)
    def constant_medium(self, boundary, density, tex): return self._call("constant_medium", boundary, density, tex)

    def constant_medium_color(self, boundary, density, rgb):
        return self.constant_medium(boundary, density, self.texture_solid(*rgb))

    def set_device_bvh(self, reference: bool):
        """Walk the recorded bvh.rs topology on the device (True) or the SAH rebuild (False, default)."""
        if self.prefix == "shim_":
            self._call("scene_set_option", 1, 1 if reference else 0)

    def world_add(self, h): return self._call("world_add", h)
    def commit(self): return self._call("commit")

    # ---- introspection
    def bvh_info(self, bvh):
        n, root, height = C.c_int(), C.c_int(), C.c_int()
        self._call("bvh_info", bvh, C.byref(n), C.byref(root), C.byref(height))
        return n.value, root.value, height.value

    def bvh_nodes(self, bvh):
        n, _, _ = self.bvh_info(bvh)
        left = np.zeros(n, np.int32); right = np.zeros(n, np.int32); parent = np.zeros(n, np.int32)
        boxes = np.zeros((n, 6), np.float32)
        self._call("bvh_nodes", bvh, left.ctypes.data, right.ctypes.data, parent.ctypes.data, boxes.ctypes.data)
        return left, right, parent, boxes
