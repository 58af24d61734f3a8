"""Host-side mirror of the reference's render entry point over the C ABI.

``Scene`` owns a committed scene handle; ``Renderer`` mirrors ``shimmer::renderer::Renderer``
(reference src/renderer.rs:22-52): ``Renderer.from_aspect_ratio(width, aspect)`` and
``render(camera, world, background, samples_per_pixel, max_depth, tile_width, tile_height,
predictors)``.  The product path is the CUDA library only; nothing here computes radiance.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import capi
from .capi import Camera, RenderParams, ShimError, Stats


class Scene(capi.SceneHandle):
    """A scene recorded through the C ABI of libshimmer_b200.so."""

    def __init__(self):
        super().__init__(capi.load_library(), "shim_")

    def bvh_from_nodes(self, left, right, root, t0=0.0, t1=1.0, with_predictor=False):
        left = np.ascontiguousarray(left, np.int32)
        right = np.ascontiguousarray(right, np.int32)
        rc = self.lib.shim_bvh_from_nodes(self.ptr, len(left), left.ctypes.data, right.ctypes.data, root, t0, t1,
                                          1 if with_predictor else 0)
        if rc < 0:
            raise ShimError(rc, self.lib.shim_last_error().decode())
        return rc

    def device_bytes(self) -> int:
        return int(self.lib.shim_scene_device_bytes(self.ptr))

    # ---- gate 1
    def trace_closest(self, rays: np.ndarray, t_min=0.001, t_max=float("inf"), seed=0, counters=False):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        prim = np.empty(n, np.int32)
        t = np.empty(n, np.float32)
        cnt = np.zeros(3, np.uint64)
        rc = self.lib.shim_trace_closest(self.ptr, rays.ctypes.data, n, t_min, t_max, seed, prim.ctypes.data, t.ctypes.data,
                                         cnt.ctypes.data if counters else None)
        if rc < 0:
            raise ShimError(rc, self.lib.shim_last_error().decode())
        return (prim, t, cnt) if counters else (prim, t)

    def trace_hit(self, rays: np.ndarray, t_min=0.001, t_max=float("inf"), seed=0, counters=False):
        """``Hittable::hit`` on the world for a batch of rays (n x 7: origin, direction, time) with the whole record:
        a structured array of ``capi.HIT_RECORD_DTYPE`` (``hittable == -1`` on a miss); with ``counters`` also
        (rays, node visits, primitive tests) as ``trace_closest`` gives them."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        out = np.empty(n, capi.HIT_RECORD_DTYPE)
        cnt = np.zeros(3, np.uint64)
        rc = self.lib.shim_trace_hit(self.ptr, rays.ctypes.data, n, t_min, t_max, seed, out.ctypes.data_as(C.POINTER(capi.HitRecord)),
                                     cnt.ctypes.data if counters else None)
        if rc < 0:
            raise ShimError(rc, self.lib.shim_last_error().decode())
        return (out, cnt) if counters else out

    def trace_hit_device(self, d_rays_ptr: int, n: int, d_out_ptr: int, t_min=0.001, t_max=float("inf"), seed=0, stream: int = 0):
        """``trace_hit`` on device buffers (e.g. ``torch.Tensor.data_ptr()``): ``d_rays_ptr`` n x 7 float32, ``d_out_ptr``
        n records of 48 bytes, 16-byte aligned.  Enqueued on ``stream``; the scene's device must be current."""
        rc = self.lib.shim_trace_hit_device(self.ptr, C.c_void_p(d_rays_ptr), n, t_min, t_max, seed,
                                            C.cast(C.c_void_p(d_out_ptr), C.POINTER(capi.HitRecord)), C.c_void_p(stream))
        if rc < 0:
            raise ShimError(rc, self.lib.shim_last_error().decode())

    def trace_occluded(self, rays: np.ndarray, t_min=0.001, t_max=float("inf"), seed=0, counters=False):
        """Is anything hit on each ray (n x 7: origin, direction, time) with t in [t_min, t_max]?  A bool array, True
        exactly where ``trace_closest`` of the same rays and seed reports a hit; the walk stops at the first hit found.
        With ``counters`` also (rays, node visits, primitive tests), never more than ``trace_closest``'s.  Visibility
        between points a and b: origin a, direction b - a, ``t_min=1e-3, t_max=1 - 1e-3``."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        out = np.empty(n, np.uint8)
        cnt = np.zeros(3, np.uint64)
        rc = self.lib.shim_trace_occluded(self.ptr, rays.ctypes.data, n, t_min, t_max, seed, out.ctypes.data,
                                          cnt.ctypes.data if counters else None)
        if rc < 0:
            raise ShimError(rc, self.lib.shim_last_error().decode())
        occ = out.view(np.bool_)
        return (occ, cnt) if counters else occ

    def trace_occluded_device(self, d_rays_ptr: int, n: int, d_out_ptr: int, t_min=0.001, t_max=float("inf"), seed=0, stream: int = 0):
        """``trace_occluded`` on device buffers (e.g. ``torch.Tensor.data_ptr()``): ``d_rays_ptr`` n x 7 float32,
        ``d_out_ptr`` n bytes (uint8 or bool: 1 = occluded).  Enqueued on ``stream``; the scene's device must be current."""
        rc = self.lib.shim_trace_occluded_device(self.ptr, C.c_void_p(d_rays_ptr), n, t_min, t_max, seed, C.c_void_p(d_out_ptr),
                                                 C.c_void_p(stream))
        if rc < 0:
            raise ShimError(rc, self.lib.shim_last_error().decode())

    # ---- render
    def render(self, camera: Camera, params: RenderParams, out: np.ndarray | None = None):
        """Blocking render into a host framebuffer; returns (H, W, 3) float32 (row 0 = bottom) and Stats.
        ``out`` may be a caller-owned C-contiguous float32 array of that shape to be reused across calls."""
        if out is None:
            out = np.empty((params.height, params.width, 3), np.float32)
        assert out.dtype == np.float32 and out.flags["C_CONTIGUOUS"] and out.shape == (params.height, params.width, 3)
        st = Stats()
        rc = self.lib.shim_render(self.ptr, C.byref(camera), C.byref(params), out.ctypes.data, C.byref(st))
        if rc < 0:
            raise ShimError(rc, self.lib.shim_last_error().decode())
        return out, st

    def render_multi(self, camera: Camera, params: RenderParams, n_devices: int = 0, devices=None, mode: str = "samples",
                     out: np.ndarray | None = None):
        """One image sharded over several devices of this process (``shim_render_multi``): sample ranges or tiles,
        per-device accumulation, one combine at the end.  Returns the host framebuffer and the summed Stats."""
        if out is None:
            out = np.empty((params.height, params.width, 3), np.float32)
        assert out.dtype == np.float32 and out.flags["C_CONTIGUOUS"] and out.shape == (params.height, params.width, 3)
        dev = None
        if devices is not None:
            dev = (C.c_int * len(devices))(*devices)
            n_devices = len(devices)
        st = Stats()
        rc = self.lib.shim_render_multi(self.ptr, C.byref(camera), C.byref(params), n_devices, dev,
                                        {"samples": capi.SHARD_SAMPLES, "tiles": capi.SHARD_TILES}[mode], out.ctypes.data, C.byref(st))
        if rc < 0:
            raise ShimError(rc, self.lib.shim_last_error().decode())
        return out, st

    def render_device(self, camera: Camera, params: RenderParams, d_out_ptr: int, stream: int = 0) -> Stats:
        """Render into a device buffer (e.g. ``torch.Tensor.data_ptr()``) on ``stream``."""
        st = Stats()
        rc = self.lib.shim_render_device(self.ptr, C.byref(camera), C.byref(params), C.c_void_p(d_out_ptr), C.byref(st),
                                         C.c_void_p(stream))
        if rc < 0:
            raise ShimError(rc, self.lib.shim_last_error().decode())
        return st


class HostFramebuffer:
    """A page-locked (H, W, 3) float32 framebuffer from ``shim_host_alloc``: ``Scene.render(..., out=fb.array)`` copies
    device -> host straight into it.  Free with ``close()`` (or let it be collected)."""

    def __init__(self, height: int, width: int):
        self.lib = capi.load_library()
        n = height * width * 3
        self.ptr = self.lib.shim_host_alloc(n)
        if not self.ptr:
            raise ShimError(-1, self.lib.shim_last_error().decode())
        self.array = np.ctypeslib.as_array((C.c_float * n).from_address(self.ptr)).reshape(height, width, 3)

    def close(self):
        if self.ptr:
            self.array = None
            self.lib.shim_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def shutdown() -> None:
    """Release every device's wavefront pool (``shim_shutdown``); scenes stay valid."""
    capi.load_library().shim_shutdown()


def pool_bytes(device: int = 0) -> int:
    return int(capi.load_library().shim_pool_bytes(device))


def make_params(width, height, spp, max_depth=50, tile_width=8, tile_height=8, background=(0.0, 0.0, 0.0), seed=0,
                sample_begin=0, sample_count=0, tile_rank=0, tile_world=0, flags=0, pool_paths=0) -> RenderParams:
    p = RenderParams()
    p.width, p.height, p.samples_per_pixel, p.max_depth = width, height, spp, max_depth
    p.tile_width, p.tile_height = tile_width, tile_height
    p.background[:] = [float(b) for b in background]
    p.seed = seed
    p.sample_begin, p.sample_count = sample_begin, sample_count
    p.tile_rank, p.tile_world = tile_rank, tile_world
    p.flags, p.pool_paths = flags, pool_paths
    return p


def image_height(image_width: int, aspect_ratio: float) -> int:
    """``Renderer::from_aspect_ratio`` (renderer.rs:34-39): f32 division, truncation."""
    return int(np.float32(image_width) / np.float32(aspect_ratio))


@dataclass
class Renderer:
    """Mirror of ``shimmer::renderer::Renderer`` (renderer.rs:22-52)."""

    image_width: int
    image_height: int

    @classmethod
    def from_aspect_ratio(cls, image_width: int, aspect_ratio: float) -> "Renderer":
        return cls(image_width, image_height(image_width, aspect_ratio))

    def render(self, camera: Camera, world: Scene, background, samples_per_pixel: int, max_depth: int,
               tile_width: int = 8, tile_height: int = 8, predictors: bool = False, seed: int = 0):
        flags = capi.RENDER_PREDICTORS if predictors else 0
        p = make_params(self.image_width, self.image_height, samples_per_pixel, max_depth, tile_width, tile_height,
                        background, seed, flags=flags)
        return world.render(camera, p)


def tile_layout(image_width, image_height, tile_width, tile_height) -> np.ndarray:
    """``Tile::tile`` (renderer.rs:242-296) -> (n, 4) int32 rows of (width, height, x0, y0)."""
    lib = capi.load_library()
    n = lib.shim_tile_layout(image_width, image_height, tile_width, tile_height, None, 0)
    if n < 0:
        raise ShimError(n, lib.shim_last_error().decode())
    out = np.zeros((n, 4), np.int32)
    lib.shim_tile_layout(image_width, image_height, tile_width, tile_height, out.ctypes.data, n)
    return out


def camera_fields(camera: Camera) -> np.ndarray:
    lib = capi.load_library()
    out = np.zeros(21, np.float32)
    lib.shim_camera_fields(C.byref(camera), out.ctypes.data)
    return out


def hrpp_hash(origin, direction) -> int:
    lib = capi.load_library()
    o = np.array(origin, np.float32)
    d = np.array(direction, np.float32)
    return int(lib.shim_hrpp_hash(o.ctypes.data, d.ctypes.data))


def write_ppm(rgb: np.ndarray, path: str | None = None) -> int:
    """``Renderer::write_ppm`` (renderer.rs:107-127): P3, no gamma, top row first."""
    lib = capi.load_library()
    a = np.ascontiguousarray(rgb, np.float32)
    h, w = a.shape[0], a.shape[1]
    return int(lib.shim_write_ppm(a.ctypes.data, w, h, path.encode() if path else None))
