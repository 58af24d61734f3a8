"""Test support: bindings for the CPU oracle (oracle/) and the hostsim harness (tests/hostsim)."""
from __future__ import annotations

import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from raytracinginoneweekendinrust_b200 import capi  # noqa: E402
from raytracinginoneweekendinrust_b200.capi import Camera, RenderParams  # noqa: E402

_P, _I, _F = C.c_void_p, C.c_int, C.c_float


class OrcRenderParams(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("max_depth", C.c_int32),
        ("tile_w", C.c_int32), ("tile_h", C.c_int32), ("background", C.c_float * 3), ("seed", C.c_uint64),
        ("sample_begin", C.c_int32), ("sample_count", C.c_int32), ("rng_fast", C.c_int32), ("iterative", C.c_int32),
        ("threads", C.c_int32), ("use_predictors", C.c_int32), ("raw_sum", C.c_int32),
    ]


class OrcStats(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("samples", C.c_uint64), ("node_visits", C.c_uint64), ("prim_tests", C.c_uint64),
                ("hrpp_tp", C.c_uint64), ("hrpp_fp", C.c_uint64), ("hrpp_none", C.c_uint64), ("seconds", C.c_double),
                ("threads", C.c_int32)]


_orc = None
_hs = None


def oracle_lib():
    global _orc
    if _orc is None:
        sys.path.insert(0, str(ROOT / "oracle"))
        import build as orc_build
        lib = C.CDLL(str(orc_build.build()))
        capi.bind_builder(lib, "orc_")
        lib.orc_aabb_hit.restype = _I
        lib.orc_aabb_hit.argtypes = [_P, _P, _P, _P, _F, _F]
        lib.orc_aabb_union.restype = None
        lib.orc_aabb_union.argtypes = [_P, _P, _P]
        lib.orc_tile_layout.restype = _I
        lib.orc_tile_layout.argtypes = [_I, _I, _I, _I, _P, _I]
        lib.orc_sphere_uv.restype = None
        lib.orc_sphere_uv.argtypes = [_F, _F, _F, _P]
        lib.orc_map_float_to_hash.restype = C.c_uint32
        lib.orc_map_float_to_hash.argtypes = [_F]
        lib.orc_hrpp_hash.restype = C.c_uint64
        lib.orc_hrpp_hash.argtypes = [_P, _P]
        lib.orc_philox.restype = None
        lib.orc_philox.argtypes = [_P, _P, _P]
        lib.orc_camera_fields.restype = None
        lib.orc_camera_fields.argtypes = [_P, _P]
        lib.orc_texture_value.restype = None
        lib.orc_texture_value.argtypes = [_P, _I, _F, _F, _P, _P]
        lib.orc_trace_closest.restype = _I
        lib.orc_trace_closest.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _I, _P, _P, _P]
        lib.orc_trace_record.restype = _I
        lib.orc_trace_record.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _P, _P]
        lib.orc_render.restype = _I
        lib.orc_render.argtypes = [_P, _P, C.POINTER(OrcRenderParams), _P, C.POINTER(OrcStats)]
        lib.orc_sample_radiance.restype = _I
        lib.orc_sample_radiance.argtypes = [_P, _P, C.POINTER(OrcRenderParams), _P, C.c_int64, _P, _P]
        lib.orc_record_path_rays.restype = C.c_int64
        lib.orc_record_path_rays.argtypes = [_P, _P, C.POINTER(OrcRenderParams), _P, C.c_int64, _P, C.c_int64]
        lib.orc_last_counters.restype = None
        lib.orc_last_counters.argtypes = [_P]
        lib.orc_predictor_stats.restype = _I
        lib.orc_predictor_stats.argtypes = [_P, _I, _P, _P]
        _orc = lib
    return _orc


def hostsim_lib():
    """CPU build of the product's __host__ __device__ math (tests/hostsim); never part of the package."""
    global _hs
    if _hs is None:
        out = ROOT / "tests" / "hostsim" / "_build" / "libhostsim.so"
        srcs = [ROOT / "tests" / "hostsim" / "hostsim.cpp",
                ROOT / "raytracinginoneweekendinrust_b200" / "csrc" / "shim_builder.cpp",
                ROOT / "raytracinginoneweekendinrust_b200" / "csrc" / "shim_scene.cpp"]
        deps = srcs + list((ROOT / "raytracinginoneweekendinrust_b200" / "csrc").glob("*.h"))
        if not out.exists() or any(d.stat().st_mtime > out.stat().st_mtime for d in deps):
            out.parent.mkdir(parents=True, exist_ok=True)
            subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", str(out),
                            *map(str, srcs)], check=True)
        lib = C.CDLL(str(out))
        capi.bind_builder(lib, "shim_")
        lib.hs_commit.restype = _I
        lib.hs_commit.argtypes = [_P]
        lib.hs_trace_closest.restype = _I
        lib.hs_trace_closest.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _P, _P, _P]
        lib.hs_trace_closest_q.restype = _I
        lib.hs_trace_closest_q.argtypes = [_P, _P, C.c_int64, _F, _F, _P, _P, _P]
        lib.hs_trace_hit.restype = _I
        lib.hs_trace_hit.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _I, _P, _P]
        lib.hs_trace_occluded.restype = _I
        lib.hs_trace_occluded.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _I, _P, _P]
        lib.hs_qnodes.restype = _I
        lib.hs_qnodes.argtypes = [_P, _P, _I]
        lib.hs_trace_closest_solo.restype = _I
        lib.hs_trace_closest_solo.argtypes = [_P, _P, C.c_int64, _F, _F, _I, _P, _P, _P]
        lib.hs_sample_radiance.restype = _I
        lib.hs_sample_radiance.argtypes = [_P, C.POINTER(Camera), C.POINTER(RenderParams), _P, C.c_int64, _P, _P]
        lib.hs_render_counts.restype = _I
        lib.hs_render_counts.argtypes = [_P, C.POINTER(Camera), C.POINTER(RenderParams), _P, C.c_int64, C.c_uint32, _I, _P]
        lib.hs_texture_value.restype = None
        lib.hs_texture_value.argtypes = [_P, _I, _F, _F, _P, _P]
        lib.hs_enable_predictors.restype = _I
        lib.hs_enable_predictors.argtypes = [_P, _I]
        lib.hs_predictor_stats.restype = None
        lib.hs_predictor_stats.argtypes = [_P, _P]
        lib.hs_philox.restype = None
        lib.hs_philox.argtypes = [_P, _P, _P]
        _hs = lib
    return _hs


class OracleScene(capi.SceneHandle):
    def __init__(self):
        super().__init__(oracle_lib(), "orc_")

    def trace_closest(self, rays, t_min=0.001, t_max=float("inf"), seed=0, counters=False, use_predictors=False):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        prim = np.empty(n, np.int32); t = np.empty(n, np.float32); cnt = np.zeros(3, np.uint64)
        rc = self.lib.orc_trace_closest(self.ptr, rays.ctypes.data, n, t_min, t_max, seed, 1 if use_predictors else 0,
                                        prim.ctypes.data, t.ctypes.data, cnt.ctypes.data)
        assert rc == 0
        return (prim, t, cnt) if counters else (prim, t)

    def trace_hit(self, rays, t_min=0.001, t_max=float("inf"), seed=0, counters=False):
        """The oracle's HitRecord and hittable id per ray, as a capi.HIT_RECORD_DTYPE array."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        out = np.empty(n, capi.HIT_RECORD_DTYPE); cnt = np.zeros(3, np.uint64)
        rc = self.lib.orc_trace_record(self.ptr, rays.ctypes.data, n, t_min, t_max, seed, out.ctypes.data, cnt.ctypes.data)
        assert rc == 0
        return (out, cnt) if counters else out

    def params(self, width, height, spp, max_depth=50, tile=(8, 8), background=(0, 0, 0), seed=0, sample_begin=0,
               sample_count=0, rng_fast=False, iterative=False, threads=0, use_predictors=False, raw_sum=False):
        p = OrcRenderParams()
        p.width, p.height, p.spp, p.max_depth = width, height, spp, max_depth
        p.tile_w, p.tile_h = tile
        p.background[:] = [float(b) for b in background]
        p.seed = seed
        p.sample_begin, p.sample_count = sample_begin, sample_count
        p.rng_fast, p.iterative, p.threads = int(rng_fast), int(iterative), threads
        p.use_predictors, p.raw_sum = int(use_predictors), int(raw_sum)
        return p

    def render(self, camera: Camera, p: OrcRenderParams):
        out = np.zeros((p.height, p.width, 3), np.float32)
        st = OrcStats()
        cam = camera.as_array15()
        rc = self.lib.orc_render(self.ptr, cam.ctypes.data, C.byref(p), out.ctypes.data, C.byref(st))
        assert rc == 0, self.lib.orc_last_error()
        return out, st

    def sample_radiance(self, camera: Camera, p: OrcRenderParams, xys):
        xys = np.ascontiguousarray(xys, np.int32).reshape(-1, 3)
        out = np.zeros((len(xys), 3), np.float32)
        rays = C.c_uint64()
        cam = camera.as_array15()
        rc = self.lib.orc_sample_radiance(self.ptr, cam.ctypes.data, C.byref(p), xys.ctypes.data, len(xys), out.ctypes.data,
                                          C.byref(rays))
        assert rc == 0
        return out, rays.value

    def last_counters(self):
        out = np.zeros(6, np.uint64)
        self.lib.orc_last_counters(out.ctypes.data)
        return dict(zip(("rays", "node_visits", "prim_tests", "hrpp_tp", "hrpp_fp", "hrpp_none"), (int(v) for v in out)))

    def record_path_rays(self, camera: Camera, p: OrcRenderParams, xys, cap):
        xys = np.ascontiguousarray(xys, np.int32).reshape(-1, 3)
        rays = np.zeros((cap, 7), np.float32)
        cam = camera.as_array15()
        n = self.lib.orc_record_path_rays(self.ptr, cam.ctypes.data, C.byref(p), xys.ctypes.data, len(xys), rays.ctypes.data, cap)
        return rays[:n]


class HostSimScene(capi.SceneHandle):
    """Product builder calls + CPU execution of the product's device math (test harness)."""

    def __init__(self):
        super().__init__(hostsim_lib(), "shim_")

    def trace_closest(self, rays, t_min=0.001, t_max=float("inf"), seed=0, counters=False):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        prim = np.empty(n, np.int32); t = np.empty(n, np.float32); cnt = np.zeros(3, np.uint64)
        self.lib.hs_trace_closest(self.ptr, rays.ctypes.data, n, t_min, t_max, seed, prim.ctypes.data, t.ctypes.data, cnt.ctypes.data)
        return (prim, t, cnt) if counters else (prim, t)

    def trace_closest_solo(self, rays, signed_nodes, t_min=0.001, t_max=float("inf")):
        """closest_hit_solo (one-Bvh worlds) on the plain or the signed node layout; returns ids, t and the counters."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        prim = np.empty(n, np.int32); t = np.empty(n, np.float32); cnt = np.zeros(3, np.uint64)
        rc = self.lib.hs_trace_closest_solo(self.ptr, rays.ctypes.data, n, t_min, t_max, 1 if signed_nodes else 0, prim.ctypes.data,
                                            t.ctypes.data, cnt.ctypes.data)
        assert rc == 0, "not a one-Bvh world"
        return prim, t, cnt

    def trace_closest_q(self, rays, t_min=0.001, t_max=float("inf")):
        """closest hit with the one Bvh object walked on its quantised nodes (QNode); returns ids, t, counters, node count."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        prim = np.empty(n, np.int32); t = np.empty(n, np.float32); cnt = np.zeros(3, np.uint64)
        nq = self.lib.hs_trace_closest_q(self.ptr, rays.ctypes.data, n, t_min, t_max, prim.ctypes.data, t.ctypes.data, cnt.ctypes.data)
        assert nq > 0, "no quantised nodes (not a one-Bvh world, or not representable)"
        return prim, t, cnt, nq

    def trace_hit(self, rays, t_min=0.001, t_max=float("inf"), seed=0, counters=False, quantised=False):
        """trace_hit_kernel's arithmetic ray by ray (capi.HIT_RECORD_DTYPE array); ``quantised``: the one Bvh object
        walked on its quantised nodes, as the kernel does for a scene that has them."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        out = np.empty(n, capi.HIT_RECORD_DTYPE); cnt = np.zeros(3, np.uint64)
        rc = self.lib.hs_trace_hit(self.ptr, rays.ctypes.data, n, t_min, t_max, seed, 1 if quantised else 0, out.ctypes.data,
                                   cnt.ctypes.data)
        assert rc == 0, "no quantised nodes (not a one-Bvh world)"
        return (out, cnt) if counters else out

    def trace_occluded(self, rays, t_min=0.001, t_max=float("inf"), seed=0, counters=False, quantised=False):
        """trace_occluded_kernel's arithmetic ray by ray (bool per ray); ``quantised``: the one Bvh object walked on its
        quantised nodes, as the kernel does for a scene that has them."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        out = np.empty(n, np.uint8); cnt = np.zeros(3, np.uint64)
        rc = self.lib.hs_trace_occluded(self.ptr, rays.ctypes.data, n, t_min, t_max, seed, 1 if quantised else 0, out.ctypes.data,
                                        cnt.ctypes.data)
        assert rc == 0, "no quantised nodes (not a one-Bvh world)"
        occ = out.view(np.bool_)
        return (occ, cnt) if counters else occ

    def enable_predictors(self, log2=16):
        return self.lib.hs_enable_predictors(self.ptr, log2)

    def predictor_stats(self):
        out = np.zeros(3, np.uint64)
        self.lib.hs_predictor_stats(self.ptr, out.ctypes.data)
        return tuple(int(v) for v in out)

    def sample_radiance(self, camera: Camera, p: RenderParams, xys):
        xys = np.ascontiguousarray(xys, np.int32).reshape(-1, 3)
        out = np.zeros((len(xys), 3), np.float32)
        rays = C.c_uint64()
        self.lib.hs_sample_radiance(self.ptr, C.byref(camera), C.byref(p), xys.ctypes.data, len(xys), out.ctypes.data, C.byref(rays))
        return out, rays.value

    def render_counts(self, camera: Camera, p: RenderParams, xys, tail_threshold=65536, generic=False):
        """(rays, node visits, primitive tests) of a counted render of the samples ``xys`` (n x 3: x, y, sample) with a
        pool that holds all of them and the endgame threshold ``tail_threshold``; ``generic``: every ray counted as
        closest_hit counts it."""
        xys = np.ascontiguousarray(xys, np.int32).reshape(-1, 3)
        out = np.zeros(3, np.uint64)
        rc = self.lib.hs_render_counts(self.ptr, C.byref(camera), C.byref(p), xys.ctypes.data, len(xys), tail_threshold,
                                       1 if generic else 0, out.ctypes.data)
        assert rc == 0
        return tuple(int(v) for v in out)


def random_xys(width, height, spp, n, seed=0):
    rs = np.random.RandomState(seed)
    return np.stack([rs.randint(0, width, n), rs.randint(0, height, n), rs.randint(0, spp, n)], axis=1).astype(np.int32)


def all_samples(width, height, spp, sample_begin=0, sample_count=0):
    """Every (x, y, sample) of a render (sample_count 0: all spp samples), in no particular order."""
    count = sample_count if sample_count > 0 else spp
    y, x, s = np.meshgrid(np.arange(height), np.arange(width), np.arange(sample_begin, sample_begin + count), indexing="ij")
    return np.stack([x.ravel(), y.ravel(), s.ravel()], axis=1).astype(np.int32)
