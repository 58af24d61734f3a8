"""Test support for the record-level parity of shim_trace_hit (tests/test_hit_records.py): the oracle with
orc_trace_hit and the hostsim harness with hs_trace_hit, each built from its unchanged source plus one added entry
point (tests/records/*.cpp) into tests/records/_build/."""
from __future__ import annotations

import ctypes as C
import subprocess
import sys

import numpy as np

import support
from support import ROOT
from raytracinginoneweekendinrust_b200 import capi

_P, _I, _F = C.c_void_p, C.c_int, C.c_float
BUILD = ROOT / "tests" / "records" / "_build"
CSRC = ROOT / "raytracinginoneweekendinrust_b200" / "csrc"

_orc = None
_hs = None


def _compile(out, srcs, deps, flags):
    if not out.exists() or any(d.stat().st_mtime > out.stat().st_mtime for d in deps):
        out.parent.mkdir(parents=True, exist_ok=True)
        subprocess.run(["g++", *flags, "-o", str(out), *map(str, srcs)], check=True)
    return out


def oracle_hit_lib():
    """oracle/shimmer_oracle.cpp + orc_trace_hit, with the oracle's flags."""
    global _orc
    if _orc is None:
        sys.path.insert(0, str(ROOT / "oracle"))
        import build as orc_build
        src = ROOT / "tests" / "records" / "oracle_hit.cpp"
        out = _compile(BUILD / "liborc_hit.so", [src], [src, orc_build.SRC], orc_build.FLAGS)
        lib = C.CDLL(str(out))
        capi.bind_builder(lib, "orc_")
        lib.orc_trace_closest.restype = _I
        lib.orc_trace_closest.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _I, _P, _P, _P]
        lib.orc_record_path_rays.restype = C.c_int64
        lib.orc_record_path_rays.argtypes = [_P, _P, C.POINTER(support.OrcRenderParams), _P, C.c_int64, _P, C.c_int64]
        lib.orc_trace_hit.restype = _I
        lib.orc_trace_hit.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _P, _P]
        _orc = lib
    return _orc


def hostsim_hit_lib():
    """tests/hostsim/hostsim.cpp + hs_trace_hit and the product's builder, with the harness's flags."""
    global _hs
    if _hs is None:
        src = ROOT / "tests" / "records" / "hostsim_hit.cpp"
        srcs = [src, CSRC / "shim_builder.cpp", CSRC / "shim_scene.cpp"]
        deps = srcs + [ROOT / "tests" / "hostsim" / "hostsim.cpp"] + list(CSRC.glob("*.h"))
        out = _compile(BUILD / "libhostsim_hit.so", srcs, deps, ["-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared"])
        lib = C.CDLL(str(out))
        capi.bind_builder(lib, "shim_")
        lib.hs_trace_closest.restype = _I
        lib.hs_trace_closest.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _P, _P, _P]
        lib.hs_trace_hit.restype = _I
        lib.hs_trace_hit.argtypes = [_P, _P, C.c_int64, _F, _F, C.c_uint64, _I, _P, _P]
        _hs = lib
    return _hs


def build():
    oracle_hit_lib()
    hostsim_hit_lib()


class OracleScene(support.OracleScene):
    """The oracle scene of tests/support.py, recorded in the library that also has orc_trace_hit."""

    def __init__(self):
        capi.SceneHandle.__init__(self, oracle_hit_lib(), "orc_")

    def trace_hit(self, rays, t_min=0.001, t_max=float("inf"), seed=0, counters=False):
        """The oracle's HitRecord and hittable id per ray, as a capi.HIT_RECORD_DTYPE array."""
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 7)
        n = rays.shape[0]
        out = np.empty(n, capi.HIT_RECORD_DTYPE); cnt = np.zeros(3, np.uint64)
        rc = self.lib.orc_trace_hit(self.ptr, rays.ctypes.data, n, t_min, t_max, seed, out.ctypes.data, cnt.ctypes.data)
        assert rc == 0
        return (out, cnt) if counters else out


class HostSimScene(support.HostSimScene):
    """The harness scene of tests/support.py, recorded in the library that also has hs_trace_hit."""

    def __init__(self):
        capi.SceneHandle.__init__(self, hostsim_hit_lib(), "shim_")

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
