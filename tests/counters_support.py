"""Test support for the counters of counted renders and ray queries (tests/test_counters.py): the hostsim harness with
hs_render_counts, built from tests/records/hostsim_counts.cpp (the unchanged occlusion harness plus that one entry point)
into tests/records/_build/."""
from __future__ import annotations

import ctypes as C

import numpy as np

import occlusion_support
import records_support
import support
from support import ROOT
from raytracinginoneweekendinrust_b200 import capi
from raytracinginoneweekendinrust_b200.capi import Camera, RenderParams

_P, _I, _F = C.c_void_p, C.c_int, C.c_float
_hs = None


def hostsim_counts_lib():
    """tests/records/hostsim_occluded.cpp + hs_render_counts and the product's builder, with the harness's flags."""
    global _hs
    if _hs is None:
        rec = ROOT / "tests" / "records"
        src = rec / "hostsim_counts.cpp"
        csrc = records_support.CSRC
        srcs = [src, csrc / "shim_builder.cpp", csrc / "shim_scene.cpp"]
        deps = srcs + [rec / "hostsim_occluded.cpp", rec / "hostsim_hit.cpp", ROOT / "tests" / "hostsim" / "hostsim.cpp"] + list(csrc.glob("*.h"))
        out = records_support._compile(records_support.BUILD / "libhostsim_counts.so", srcs, deps,
                                       ["-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared"])
        lib = C.CDLL(str(out))
        capi.bind_builder(lib, "shim_")
        lib.hs_trace_closest.restype = _I
        lib.hs_trace_closest.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _P, _P, _P]
        lib.hs_trace_hit.restype = _I
        lib.hs_trace_hit.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _I, _P, _P]
        lib.hs_trace_occluded.restype = _I
        lib.hs_trace_occluded.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _I, _P, _P]
        lib.hs_sample_radiance.restype = _I
        lib.hs_sample_radiance.argtypes = [_P, C.POINTER(Camera), C.POINTER(RenderParams), _P, C.c_int64, _P, _P]
        lib.hs_render_counts.restype = _I
        lib.hs_render_counts.argtypes = [_P, C.POINTER(Camera), C.POINTER(RenderParams), _P, C.c_int64, C.c_uint32, _I, _P]
        _hs = lib
    return _hs


def build():
    hostsim_counts_lib()


class HostSimScene(occlusion_support.HostSimScene, records_support.HostSimScene):
    """The harness scene of tests/support.py with all three ray queries and hs_render_counts in one library."""

    def __init__(self):
        capi.SceneHandle.__init__(self, hostsim_counts_lib(), "shim_")

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


def all_samples(width, height, spp, sample_begin=0, sample_count=0):
    """Every (x, y, sample) of a render (sample_count 0: all spp samples), in no particular order."""
    count = sample_count if sample_count > 0 else spp
    y, x, s = np.meshgrid(np.arange(height), np.arange(width), np.arange(sample_begin, sample_begin + count), indexing="ij")
    return np.stack([x.ravel(), y.ravel(), s.ravel()], axis=1).astype(np.int32)
