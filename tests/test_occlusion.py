"""Occlusion, the any-hit query (shim_trace_occluded): is anything hit on the ray between t_min and t_max?

Its walk is the closest-hit walk cut off at the first accepted hit, so for every ray, seed and interval
``occluded == (trace_closest(...).prim_id >= 0)`` bit for bit, with no more node visits or primitive tests.  On the CPU
the product's device arithmetic (hs_trace_occluded in tests/hostsim: closest_hit<..., ANY = true>) is checked against its
own closest-hit query (exact) and against the oracle's ``prim >= 0``.  With -m gpu the kernel is checked the same way
against shim_trace_closest (exact, media included: both draw the same device logf) and against the oracle, where media
scenes may also differ by gate 1b's number of flipped accepts (device logf).

Against the oracle one more exception is allowed, and it is the closest-hit query's, not this one's: a segment between
two points of one axis-aligned face lies in that face's plane (a direction component is exactly 0).  There the device
closest-hit walk can miss where the oracle reports a hit at t = NaN, and the occlusion query answers as the walk does.

Rays: the path rays and random rays of tests/test_hit_records.py with t in [0.001, inf), and segments between two
recorded hit points a and b (origin a, direction b - a, t in [1e-3, 1 - 1e-3]), the visibility idiom of the header."""
import numpy as np
import pytest

import support
import test_gpu_parity as T
import test_hit_records as HR
from fuzz_scenes import build_random_scene, random_rays
from raytracinginoneweekendinrust_b200 import api, capi, scenes

SEG_T = (1e-3, 1.0 - 1e-3)


def segments(points, n, seed):
    """n segments between random pairs of the points (origin a, direction b - a, time in [0, 1)); pairs closer than
    1e-2 are dropped."""
    rs = np.random.RandomState(seed)
    a, b = rs.randint(0, len(points), n), rs.randint(0, len(points), n)
    d = points[b] - points[a]
    keep = np.linalg.norm(d, axis=1) > 1e-2
    seg = np.empty((keep.sum(), 7), np.float32)
    seg[:, 0:3] = points[a[keep]]
    seg[:, 3:6] = d[keep]
    seg[:, 6] = rs.uniform(0, 1, keep.sum())
    return seg


def hit_points(o, rays, seed):
    """The oracle's hit points of the rays that hit something."""
    rec = o.trace_hit(rays, seed=seed)
    return rec["point"][rec["hittable"] >= 0]


def in_axis_plane(rays):
    return (rays[:, 3:6] == 0).any(axis=1)


def assert_matches_oracle(occ, p_ref, rays, what, allowed=0):
    """occ equals the oracle's prim >= 0 up to ``allowed`` flips, plus at most 0.5 % of the rays that lie in an axis
    plane (see the module docstring)."""
    off = occ != (p_ref >= 0)
    plane = in_axis_plane(rays)
    assert off.sum() <= allowed + min(int((off & plane).sum()), len(rays) // 200), \
        f"{what}: {off.sum()} differ from the oracle, {(off & ~plane).sum()} of them not in an axis plane"


def check_against_closest(h, o, rays, t_min, t_max, seed, what):
    """The harness's occlusion answer equals its own closest-hit query's prim >= 0 and the oracle's (see the module
    docstring); its counts are at most the closest-hit query's.  Returns the answer and both count triples."""
    occ, cnt = h.trace_occluded(rays, t_min, t_max, seed=seed, counters=True)
    p_ref, _ = o.trace_closest(rays, t_min, t_max, seed=seed)
    p, _, cnt_closest = h.trace_closest(rays, t_min, t_max, seed=seed, counters=True)
    np.testing.assert_array_equal(occ, p >= 0, err_msg=what + ": against trace_closest")
    assert_matches_oracle(occ, p_ref, rays, what)
    assert cnt[0] == cnt_closest[0] == len(rays)
    assert cnt[1] <= cnt_closest[1] and cnt[2] <= cnt_closest[2], f"{what}: {cnt} vs {cnt_closest}"
    return occ, cnt, cnt_closest


# ------------------------------------------------------------------------------------------------ CPU (hostsim)
@pytest.mark.parametrize("reference_tree", [False, True])
@pytest.mark.parametrize("name", list(scenes.SCENES))
def test_occluded_is_closest_hit_found(name, reference_tree):
    kw = T.SMALL.get(name, {})
    o, h = support.OracleScene(), support.HostSimScene()
    info = scenes.build(o, name, seed=1, **kw)
    h.set_device_bvh(reference_tree)
    scenes.build(h, name, seed=1, **kw)
    rays = HR.scene_rays(o, name, info)
    occ, cnt, cnt_closest = check_against_closest(h, o, rays, 0.001, np.inf, 13, name)
    assert 0.1 < occ.mean() < 0.995, occ.mean()
    seg = segments(hit_points(o, rays, 13), 6000, seed=5)
    occ_s, _, _ = check_against_closest(h, o, seg, *SEG_T, 17, name + " segments")
    if name != "earth":   # one sphere: a chord between two of its points is never occluded
        assert 0.02 < occ_s.mean() < 0.98, occ_s.mean()
    if name == "random-spheres":   # most rays hit, and the first sphere found is rarely the last one tested
        assert cnt[1] < cnt_closest[1]


@pytest.mark.parametrize("name", ["bunny", "gargoyle", "igea-hrpp"])
def test_quantised_mesh_walk(name):
    """A mesh among the Cornell rects walked on its quantised nodes, as the kernel does for such a scene, against the
    closest-hit walk on the same nodes (the harness's hs_trace_closest_q; these scenes have no media, so the seed does
    not matter)."""
    kw = T.SMALL.get(name, {})
    o, h, hq = support.OracleScene(), support.HostSimScene(), support.HostSimScene()
    info = scenes.build(o, name, seed=1, **kw)
    scenes.build(h, name, seed=1, **kw)
    scenes.build(hq, name, seed=1, **kw)
    rays = HR.scene_rays(o, name, info)
    seg = segments(hit_points(o, rays, 2), 6000, seed=6)
    for r, (t_min, t_max), what in ((rays, (0.001, np.inf), "path and random rays"), (seg, SEG_T, "segments")):
        occ, cnt = h.trace_occluded(r, t_min, t_max, seed=2, counters=True, quantised=True)
        p, _, cnt_closest, _ = hq.trace_closest_q(r, t_min, t_max)
        np.testing.assert_array_equal(occ, p >= 0, err_msg=f"{name} {what}: against the quantised closest-hit walk")
        np.testing.assert_array_equal(occ, h.trace_occluded(r, t_min, t_max, seed=2), err_msg=f"{name} {what}: exact nodes")
        assert_matches_oracle(occ, o.trace_closest(r, t_min, t_max, seed=2)[0], r, f"{name} {what}")
        assert cnt[0] == cnt_closest[0] and cnt[1] <= cnt_closest[1] and cnt[2] <= cnt_closest[2], f"{name} {what}: {cnt} vs {cnt_closest}"
        assert occ.any() and not occ.all()


@pytest.mark.parametrize("reference_tree", [False, True])
@pytest.mark.parametrize("seed", range(6))
def test_fuzz_scenes(seed, reference_tree):
    o, h = support.OracleScene(), support.HostSimScene()
    build_random_scene(o, seed)
    h.set_device_bvh(reference_tree)
    build_random_scene(h, seed)
    rays = random_rays(seed, 6000)
    occ, _, _ = check_against_closest(h, o, rays, 0.001, np.inf, seed, f"fuzz seed {seed}")
    assert occ.sum() > 1000
    seg = segments(hit_points(o, rays, seed), 3000, seed=seed)
    check_against_closest(h, o, seg, *SEG_T, seed, f"fuzz seed {seed} segments")


@pytest.mark.parametrize("name", ["random-spheres", "cornell", "cornell-smoke", "showcase"])
def test_interval_ends_at_the_hit(name):
    """t_max equal to the closest hit's t (bit for bit) and one ulp below it: the same answer as trace_closest's with
    that t_max, ray by ray (each ray alone in its batch, so the Philox key is the same in both queries).  The oracle is
    left out: at a bound equal to the hit's t the closest-hit query itself can answer otherwise than the oracle (one
    showcase ray here), a closest-hit parity question outside this query."""
    kw = T.SMALL.get(name, {})
    o, h = support.OracleScene(), support.HostSimScene()
    info = scenes.build(o, name, seed=1, **kw)
    scenes.build(h, name, seed=1, **kw)
    rays = HR.scene_rays(o, name, info, n_paths=200, cap=2000)
    rs = np.random.RandomState(3)
    answers = []
    for i in rs.permutation(len(rays))[:200]:
        r = rays[i:i + 1]
        p, t = h.trace_closest(r, seed=4)
        if p[0] < 0:
            continue
        for t_max in (t[0], np.nextafter(t[0], np.float32(-np.inf))):
            occ = h.trace_occluded(r, t_max=t_max, seed=4)
            p_edge, _ = h.trace_closest(r, t_max=t_max, seed=4)
            assert occ[0] == (p_edge[0] >= 0), (i, t_max)
            answers.append(bool(occ[0]))
    assert len(answers) > 100
    assert 0 < sum(answers) < len(answers)


def test_empty_batch_and_misses():
    h = support.HostSimScene()
    scenes.build(h, "random-spheres", seed=1)
    rays = np.array([[0, 50, 0, 0, 1, 0, 0], [0, 2000, 0, 1, 0.5, 0, 0.5], [0, 1, -30, 0, 0, 1, 0]], np.float32)
    np.testing.assert_array_equal(h.trace_occluded(rays), [False, False, True])
    assert len(h.trace_occluded(np.zeros((0, 7), np.float32))) == 0


def test_state_and_argument_errors_without_a_commit():
    """An uncommitted scene is a state error for both variants, a null scene an invalid argument; nothing is written."""
    s = api.Scene()
    for call in (lambda: s.trace_occluded(np.zeros((1, 7), np.float32)), lambda: s.trace_occluded_device(0, 1, 0)):
        with pytest.raises(capi.ShimError) as e:
            call()
        assert e.value.code == -4 and "not committed" in e.value.message
    lib = capi.load_library()
    rays = np.zeros((1, 7), np.float32)
    out = np.full(1, 7, np.uint8)
    cnt = np.full(3, 9, np.uint64)
    assert lib.shim_trace_occluded(None, rays.ctypes.data, 1, 0.001, np.inf, 0, out.ctypes.data, cnt.ctypes.data) == -1
    assert lib.shim_trace_occluded(s.ptr, rays.ctypes.data, 1, 0.001, np.inf, 0, out.ctypes.data, cnt.ctypes.data) == -4
    assert lib.shim_trace_occluded_device(None, None, 1, 0.001, np.inf, 0, None, None) == -1
    assert (out == 7).all() and (cnt == 9).all()


@pytest.mark.skipif(HR._has_cuda(), reason="needs a machine without a CUDA device")
def test_no_cpu_fallback_without_a_device():
    """Without a device the scene cannot be committed (SHIM_ERR_CUDA), so the query reports the state error and leaves
    the output as it was instead of computing anything on the CPU."""
    s = api.Scene()
    scenes.random_spheres(s, seed=1)
    with pytest.raises(capi.ShimError) as e:
        s.commit()
    assert e.value.code == -3 and "no CPU fallback" in e.value.message
    out = np.full(4, 7, np.uint8)
    lib = capi.load_library()
    rays = np.zeros((4, 7), np.float32)
    assert lib.shim_trace_occluded(s.ptr, rays.ctypes.data, 4, 0.001, np.inf, 0, out.ctypes.data, None) == -4
    assert (out == 7).all()


def test_rust_wrapper_has_the_query():
    """The -sys declarations are checked against the header by tests/test_rust_binding.py; this is the safe wrapper."""
    wrapper = (support.ROOT / "rust" / "shimmer-b200" / "src" / "lib.rs").read_text()
    assert "pub fn trace_occluded(&mut self, rays: &[f32], t_min: f32, t_max: f32, seed: u64) -> Result<Vec<bool>>" in wrapper


# ------------------------------------------------------------------------------------------------ GPU
def gpu_rays(o, name, info, n_xy=6000, cap=60000, seed=1):
    cam = T.CAMERAS[name]
    po = o.params(160, 120, 4, 50, background=info.background, seed=3, iterative=True)
    return o.record_path_rays(cam, po, support.random_xys(160, 120, 4, n_xy, seed=seed), cap)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(scenes.SCENES))
def test_gpu_occluded_is_closest_hit_found(name):
    g, o, info = HR.build_pair(name)
    rays = gpu_rays(o, name, info)
    assert len(rays) > 6000
    seg = segments(hit_points(o, rays, 3), 30000, seed=8)
    for r, (t_min, t_max), what in ((rays, (0.001, np.inf), "path rays"), (seg, SEG_T, "segments")):
        occ = g.trace_occluded(r, t_min, t_max, seed=3)
        p, _ = g.trace_closest(r, t_min, t_max, seed=3)
        np.testing.assert_array_equal(occ, p >= 0, err_msg=f"{name} {what}: against shim_trace_closest")
        # volumes draw ln(U): device logf differs from glibc by an ulp, which can flip an accept at a boundary
        assert_matches_oracle(occ, o.trace_closest(r, t_min, t_max, seed=3)[0], r, f"{name} {what}",
                              0 if name not in HR.MEDIA_SCENES else max(2, len(r) // 20000))
        # the counted walk (exact nodes): the same answers, never more work than the closest-hit query's counted walk
        occ_c, cnt = g.trace_occluded(r, t_min, t_max, seed=3, counters=True)
        _, _, cnt_closest = g.trace_closest(r, t_min, t_max, seed=3, counters=True)
        np.testing.assert_array_equal(occ, occ_c, err_msg=f"{name} {what}: counted walk")
        assert cnt[0] == cnt_closest[0] == len(r)
        assert cnt[1] <= cnt_closest[1] and cnt[2] <= cnt_closest[2], f"{name} {what}: {cnt} vs {cnt_closest}"
        assert occ.any() and not occ.all()


@pytest.mark.gpu
def test_gpu_device_variant_on_a_side_stream():
    import torch
    g, o, info = HR.build_pair("cornell-smoke")
    cam = T.CAMERAS["cornell-smoke"]
    po = o.params(96, 96, 4, 50, background=info.background, seed=9, iterative=True)
    rays = o.record_path_rays(cam, po, support.random_xys(96, 96, 4, 3000, seed=3), 30000)
    n = len(rays)
    host = g.trace_occluded(rays, seed=9)
    d_rays = torch.from_numpy(rays).cuda()
    d_out = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        g.trace_occluded_device(d_rays.data_ptr(), n, d_out.data_ptr(), seed=9, stream=side.cuda_stream)
    side.synchronize()
    np.testing.assert_array_equal(d_out.cpu().numpy(), host.astype(np.uint8))
    # argument rules of the device variant; nothing is written
    d_out.fill_(7)
    for bad in (lambda: g.trace_occluded_device(d_rays.data_ptr(), -1, d_out.data_ptr()),
                lambda: g.trace_occluded_device(0, n, d_out.data_ptr()),
                lambda: g.trace_occluded_device(d_rays.data_ptr(), n, 0)):
        with pytest.raises(capi.ShimError) as e:
            bad()
        assert e.value.code == -1
    g.trace_occluded_device(0, 0, 0)                                                                # n == 0: no-op
    torch.cuda.synchronize()
    assert (d_out == 7).all().item()
    occ, cnt = g.trace_occluded(np.zeros((0, 7), np.float32), counters=True)
    assert len(occ) == 0 and list(cnt) == [0, 0, 0]


@pytest.mark.gpu
def test_gpu_grid_stride_batch():
    """More rays than the grid has threads (148 SMs x 2048), a count that is not a multiple of the block size:
    every answer is written and right.  Rays of a scene without media repeat with the period of the tiling."""
    g, o, info = HR.build_pair("random-spheres")
    cam = T.CAMERAS["random-spheres"]
    po = o.params(160, 120, 4, 50, background=info.background, seed=5, iterative=True)
    base = o.record_path_rays(cam, po, support.random_xys(160, 120, 4, 4000, seed=2), 40000)
    n = 700001
    assert n % 256 and n > 148 * 2048
    rays = np.resize(base, (n, 7))
    occ = g.trace_occluded(rays, seed=5)
    p_ref, _ = o.trace_closest(base, seed=5)
    np.testing.assert_array_equal(occ, (p_ref >= 0)[np.arange(n) % len(base)])
