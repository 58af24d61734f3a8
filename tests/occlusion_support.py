"""Test support for the occlusion query (tests/test_occlusion.py): the hostsim harness with hs_trace_occluded, built from
tests/records/hostsim_occluded.cpp (the unchanged record harness plus that one entry point) into tests/records/_build/."""
from __future__ import annotations

import ctypes as C

import numpy as np

import records_support
import support
from support import ROOT
from raytracinginoneweekendinrust_b200 import capi

_P, _I, _F = C.c_void_p, C.c_int, C.c_float
_hs = None


def hostsim_occluded_lib():
    """tests/records/hostsim_hit.cpp + hs_trace_occluded and the product's builder, with the harness's flags."""
    global _hs
    if _hs is None:
        rec = ROOT / "tests" / "records"
        src = rec / "hostsim_occluded.cpp"
        csrc = records_support.CSRC
        srcs = [src, csrc / "shim_builder.cpp", csrc / "shim_scene.cpp"]
        deps = srcs + [rec / "hostsim_hit.cpp", ROOT / "tests" / "hostsim" / "hostsim.cpp"] + list(csrc.glob("*.h"))
        out = records_support._compile(records_support.BUILD / "libhostsim_occluded.so", srcs, deps,
                                       ["-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared"])
        lib = C.CDLL(str(out))
        capi.bind_builder(lib, "shim_")
        lib.hs_trace_closest.restype = _I
        lib.hs_trace_closest.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _P, _P, _P]
        lib.hs_trace_occluded.restype = _I
        lib.hs_trace_occluded.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _I, _P, _P]
        _hs = lib
    return _hs


def build():
    hostsim_occluded_lib()


class HostSimScene(support.HostSimScene):
    """The harness scene of tests/support.py, recorded in the library that also has hs_trace_occluded."""

    def __init__(self):
        capi.SceneHandle.__init__(self, hostsim_occluded_lib(), "shim_")

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
