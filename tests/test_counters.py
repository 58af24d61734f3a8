"""The counters of counted renders (SHIM_RENDER_COUNT_NODES) and of the counted ray queries: rays, node visits and
primitive tests.  bench.py divides node visits and primitive tests by rays to get its instruction budget, so they are
held to an exact CPU count here.

The reference is hs_render_counts in tests/hostsim/hostsim.cpp: the paths of hs_sample_radiance, every ray counted
as the kernel that traces it in the render counts it.  A counted render walks the exact 64-byte nodes:
  - a world with one Bvh among plain objects and no medium goes through the mesh pipeline (wf_bvh1_list + wf_bvh1_walk):
    one primitive test per list object, the root's two child boxes against the closest list hit as a gate that is not a
    node visit, and if it passes the walk from the root bounded by that t;
  - every other world through wf_extend: closest_hit's counts (the list in order, each Bvh walked up to the hit so far);
  - the endgame (wf_tail), which follows the last <= SHIM_TAIL (65536) paths to their end, counts as closest_hit does.
    With a pool that holds every sample, iteration j traces exactly the bounce-j rays, so the endgame's first bounce is
    the first b >= 1 that at most that many paths reach.

On the CPU the harness is checked against the oracle's rays, against hs_trace_closest's counters on the same rays and,
on the worlds without a Bvh or a medium, against a closed form.  With -m gpu the render's and the queries' counters must
equal the harness exactly, except on the two media scenes: there the device logf and glibc's can differ by an ulp and
flip a free-path accept (the allowance of test_gpu_parity.py), which changes the rest of that path."""
import os
from unittest import mock

import numpy as np
import pytest

import support
import test_gpu_parity as T
from raytracinginoneweekendinrust_b200 import api, capi, scenes

NAMES = list(scenes.SCENES)
MEDIA = ("cornell-smoke", "showcase")
FLAT = ("two-spheres", "marble", "earth", "simple-lights", "cornell")     # world lists without a Bvh or a medium
MESH = ("bunny", "gargoyle", "igea-hrpp")                                  # one Bvh among the Cornell rects: the mesh pipeline
COUNT = capi.RENDER_COUNT_NODES
TAIL = 65536                                                               # the render's default endgame threshold


def harness(name, reference_tree=False):
    h = support.HostSimScene()
    h.set_device_bvh(reference_tree)
    info = scenes.build(h, name, seed=1, **T.SMALL.get(name, {}))
    return h, info


def counts(st):
    return int(st.rays), int(st.node_visits), int(st.prim_tests)


# ---------------------------------------------------------------------------------------------------- CPU: the harness
@pytest.mark.parametrize("name", NAMES)
def test_harness_traces_the_integrators_rays(name):
    """hs_render_counts follows the paths of hs_sample_radiance and of the oracle's integrator: the same number of rays."""
    o = support.OracleScene()
    info = scenes.build(o, name, seed=1, **T.SMALL.get(name, {}))
    h, _ = harness(name)
    cam = T.CAMERAS[name]
    W, H, spp = 120, 90, 4
    xys = support.random_xys(W, H, spp, 1500, seed=4)
    p = api.make_params(W, H, spp, 50, background=info.background, seed=13)
    _, n_orc = o.sample_radiance(cam, o.params(W, H, spp, 50, background=info.background, seed=13, iterative=True), xys)
    _, n_hs = h.sample_radiance(cam, p, xys)
    for threshold in (0, 300, TAIL):
        assert h.render_counts(cam, p, xys, threshold)[0] == n_hs == n_orc


@pytest.mark.parametrize("reference_tree", [False, True])
@pytest.mark.parametrize("name", [n for n in NAMES if n not in MEDIA])
def test_harness_generic_counts_equal_trace_closest(name, reference_tree):
    """Counted as closest_hit counts them, the paths' node visits and primitive tests are hs_trace_closest's counters
    summed over the same rays (the oracle's recorded path rays; the device drops a NaN ray without walking it)."""
    o = support.OracleScene()
    info = scenes.build(o, name, seed=1, **T.SMALL.get(name, {}))
    h, _ = harness(name, reference_tree)
    cam = T.CAMERAS[name]
    W, H, spp = 120, 90, 4
    xys = support.random_xys(W, H, spp, 1500, seed=4)
    cap = 200000
    rays = o.record_path_rays(cam, o.params(W, H, spp, 50, background=info.background, seed=13, iterative=True), xys, cap)
    assert len(rays) < cap
    finite = rays[~np.isnan(rays).any(axis=1)]
    _, _, cnt = h.trace_closest(finite, counters=True)
    n, nodes, prims = h.render_counts(cam, api.make_params(W, H, spp, 50, background=info.background, seed=13), xys, generic=True)
    assert (nodes, prims) == (int(cnt[1]), int(cnt[2]))
    assert n >= len(finite)
    if name in MESH:   # the mesh pipeline's counts: list and gate first, so never more than closest_hit's
        _, m_nodes, m_prims = h.render_counts(cam, api.make_params(W, H, spp, 50, background=info.background, seed=13), xys, tail_threshold=0)
        assert 0 < m_nodes <= nodes and m_prims <= prims


@pytest.mark.parametrize("name", FLAT)
def test_flat_world_counts_in_closed_form(name):
    """A world list without a Bvh makes one primitive test per object for every ray it walks and visits no node:
    prim_tests = (rays - NaN rays) x objects, rays from the oracle's integrator."""
    o = support.OracleScene()
    info = scenes.build(o, name, seed=1)
    h = support.HostSimScene()
    objects = []
    add = h.world_add
    h.world_add = lambda obj: (objects.append(obj), add(obj))[1]
    scenes.build(h, name, seed=1)
    cam = T.CAMERAS[name]
    W, H, spp = 120, 90, 4
    xys = support.random_xys(W, H, spp, 1500, seed=4)
    rays = o.record_path_rays(cam, o.params(W, H, spp, 50, background=info.background, seed=13, iterative=True), xys, 200000)
    walked = int((~np.isnan(rays).any(axis=1)).sum())
    for threshold in (0, TAIL):
        n, nodes, prims = h.render_counts(cam, api.make_params(W, H, spp, 50, background=info.background, seed=13), xys, threshold)
        assert nodes == 0 and prims == walked * len(objects) and n >= walked, (n, nodes, prims, walked, len(objects))


# ---------------------------------------------------------------------------------------------------- GPU: counted renders
def assert_counts_match_harness(name, got, want):
    """Exact, except on media scenes: a device logf flip changes the rest of one path, so its rays and what they walk.
    The rays may differ as much as test_gpu_parity.py allows against the oracle (0.5 %).  Node visits and primitive
    tests may differ by twice the rays' relative difference plus 1e-4: the rays a flip adds or removes cost about what
    the average ray costs (measured on a B200: on showcase 64x48x4, rays -6.4e-4, node visits -6.1e-4, primitive tests
    -6.9e-4; on cornell-smoke 320x240x2, rays -1.4e-5, primitive tests -1.3e-5)."""
    if name not in MEDIA:
        assert got == want, f"(rays, node visits, primitive tests): render {got}, harness {want}"
        return
    rel_rays = abs(got[0] - want[0]) / want[0]
    rel = [abs(g - w) / max(w, 1) for g, w in zip(got[1:], want[1:])]
    assert rel_rays <= 0.005 and max(rel) <= 2 * rel_rays + 1e-4, f"(rays, node visits, primitive tests): render {got}, harness {want}"


def assert_image_matches_oracle(name, img, st, ref, so, W, H):
    """test_render_matches_oracle_same_stream's allowances: libm-dependent scenes may have a few outlier pixels."""
    diff = np.abs(img - ref)
    outlier = diff.max(axis=2) > 1e-3
    allowed = 0 if name in ("random-spheres", "two-spheres", "cornell", "bunny", "gargoyle", "igea-hrpp") else max(2, W * H // 500)
    assert outlier.sum() <= allowed, f"{outlier.sum()} outlier pixels"
    assert float(np.sqrt(np.mean(diff[~outlier] ** 2))) <= 1e-5
    assert abs(int(st.rays) - int(so.rays)) <= (0 if allowed == 0 else max(8, so.rays // 200)), (st.rays, so.rays)


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_gpu_counted_render(name):
    """A counted render: the uncounted render's rays, the oracle's image, and the harness's counts.  12 288 samples:
    the endgame starts right after the camera rays."""
    g, o, info = T.build_pair(name)
    h, _ = harness(name)
    cam = T.CAMERAS[name]
    W, H, spp = 64, 48, 4
    p = api.make_params(W, H, spp, 50, background=info.background, seed=5, flags=COUNT)
    img, st = g.render(cam, p)
    plain, st0 = g.render(cam, api.make_params(W, H, spp, 50, background=info.background, seed=5))
    assert st.extend_variant == (1 if name in MESH else 0)     # wf_bvh1_list / _walk on exact nodes, or wf_extend
    assert st.rays == st0.rays
    np.testing.assert_allclose(img, plain, rtol=2e-5, atol=2e-6)
    ref, so = o.render(cam, o.params(W, H, spp, 50, background=info.background, seed=5))
    assert_image_matches_oracle(name, img, st, ref, so, W, H)
    assert_counts_match_harness(name, counts(st), h.render_counts(cam, p, support.all_samples(W, H, spp), TAIL))


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_gpu_counted_render_endgame_mid_render(name):
    """153 600 samples: the endgame starts after several full iterations."""
    g, o, info = T.build_pair(name)
    h, _ = harness(name)
    cam = T.CAMERAS[name]
    W, H, spp = 320, 240, 2
    p = api.make_params(W, H, spp, 50, background=info.background, seed=7, flags=COUNT)
    _, st = g.render(cam, p)
    assert st.iterations > 1 or name == "earth"   # a lone sphere: at most 65 536 paths outlive the camera rays
    assert_counts_match_harness(name, counts(st), h.render_counts(cam, p, support.all_samples(W, H, spp), TAIL))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["random-spheres", "cornell", "bunny", "showcase"])
def test_gpu_counts_do_not_depend_on_how_the_render_runs(name):
    """The endgame threshold (the harness gets the same one), the host-driven loop, the scene in global memory and a
    pool smaller than the sample count.  With such a pool the endgame's first bounce differs from path to path, so that
    render is compared with the default-pool render: without an endgame, and on worlds that count every ray as
    closest_hit does also with it."""
    g, o, info = T.build_pair(name)
    h, _ = harness(name)
    cam = T.CAMERAS[name]
    W, H, spp = 64, 48, 4
    xys = support.all_samples(W, H, spp)
    p = api.make_params(W, H, spp, 50, background=info.background, seed=5, flags=COUNT)
    small = api.make_params(W, H, spp, 50, background=info.background, seed=5, flags=COUNT, pool_paths=2048)
    _, base = g.render(cam, p)
    runs = {}
    for env, threshold in (({}, TAIL), ({"SHIM_TAIL": "0"}, 0), ({"SHIM_TAIL": "4096"}, 4096), ({"SHIM_NO_GRAPH": "1"}, TAIL),
                           ({"SHIM_NO_SMEM": "1"}, TAIL), ({"SHIM_NO_GRAPH": "1", "SHIM_TAIL": "0"}, 0)):
        with mock.patch.dict(os.environ, env):
            _, st = g.render(cam, p)
        runs[str(env)] = counts(st)
        if name in MEDIA:   # every run draws the same device logf and counts every ray as closest_hit does
            assert counts(st) == counts(base), env
        else:
            assert counts(st) == h.render_counts(cam, p, xys, threshold), env
    with mock.patch.dict(os.environ, {"SHIM_TAIL": "0"}):
        _, st = g.render(cam, small)
    assert st.iterations > 6
    assert counts(st) == runs[str({"SHIM_TAIL": "0"})]
    if name not in MESH:
        _, st = g.render(cam, small)
        assert counts(st) == counts(base)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["random-spheres", "cornell-smoke", "bunny"])
def test_gpu_shard_counts_add_up(name):
    """Sample-range shards and tile shards count what the full render counts, through shim_render and through
    shim_render_multi on one device and on two when two are present.  Each shard has its own endgame, so the mesh
    scene, whose endgame counts differently from its iterations, runs without one here."""
    g, o, info = T.build_pair(name)
    cam = T.CAMERAS[name]
    W, H, spp = 72, 56, 6

    def params(**kw):
        return api.make_params(W, H, spp, 50, background=info.background, seed=11, flags=COUNT | capi.RENDER_RAW_SUM, **kw)

    with mock.patch.dict(os.environ, {"SHIM_TAIL": "0"} if name in MESH else {}):
        full = counts(g.render(cam, params())[1])
        parts = [counts(g.render(cam, params(sample_begin=b, sample_count=c))[1]) for b, c in ((0, 2), (2, 1), (3, 3))]
        assert tuple(map(sum, zip(*parts))) == full
        tiles = [counts(g.render(cam, params(tile_rank=r, tile_world=3))[1]) for r in range(3)]
        assert tuple(map(sum, zip(*tiles))) == full
        n_dev = _n_devices()
        for devices in ([0], [0, 1]) if n_dev > 1 else ([0],):
            for mode in ("samples", "tiles"):
                _, st = g.render_multi(cam, params(), devices=devices, mode=mode)
                assert counts(st) == full, (devices, mode)


def _n_devices():
    import torch
    return torch.cuda.device_count()


# ---------------------------------------------------------------------------------------------------- GPU: ray queries
MISS = np.array([1e6, 1e6, 1e6, 1.0, 1.0, 1.0, 0.0], np.float32)   # starts far outside every scene and leaves it


def _query_counts(s, rays, seed):
    _, _, c = s.trace_closest(rays, seed=seed, counters=True)
    _, ch = s.trace_hit(rays, seed=seed, counters=True)
    _, co = s.trace_occluded(rays, seed=seed, counters=True)
    return {"closest": tuple(map(int, c)), "hit": tuple(map(int, ch)), "occluded": tuple(map(int, co))}


def _assert_query_counts(g, h, rays, seed, media):
    """On media scenes the rays whose closest hit flips (device logf, at most gate 1's allowance) are replaced by a ray
    that misses the scene at the same index (the Philox key of every other ray stays), then the counts are exact."""
    if media:
        p_g, _ = g.trace_closest(rays, seed=seed)
        p_h, _ = h.trace_closest(rays, seed=seed)
        flip = p_g != p_h
        assert flip.sum() <= max(2, len(rays) // 20000), f"{flip.sum()} flipped ids"
        rays = rays.copy()
        rays[flip] = MISS
    got, want = _query_counts(g, rays, seed), _query_counts(h, rays, seed)
    assert got == want, f"device {got}, harness {want}"
    assert got["occluded"][1] <= got["closest"][1] and got["occluded"][2] <= got["closest"][2]


@pytest.mark.gpu
@pytest.mark.parametrize("reference_tree", [False, True])
@pytest.mark.parametrize("name", NAMES)
def test_gpu_query_counters_equal_harness(name, reference_tree):
    """shim_trace_closest / _hit / _occluded with counters: the exact nodes' walk, counted as hs_trace_* count it, on the
    path rays of the scene (the mesh scenes too: a counted query does not walk the quantised nodes)."""
    g = api.Scene()
    g.set_device_bvh(reference_tree)
    info = scenes.build(g, name, seed=1, **T.SMALL.get(name, {}))
    h, _ = harness(name, reference_tree)
    o = support.OracleScene()
    scenes.build(o, name, seed=1, **T.SMALL.get(name, {}))
    cam = T.CAMERAS[name]
    W, H, spp = 160, 120, 4
    rays = o.record_path_rays(cam, o.params(W, H, spp, 50, background=info.background, seed=3, iterative=True),
                              support.random_xys(W, H, spp, 6000, seed=1), 60000)
    _assert_query_counts(g, h, rays, 3, name in MEDIA)


@pytest.mark.gpu
def test_gpu_query_counters_over_grid_passes():
    """More rays than one pass of the grid covers (148 SMs x 2048 threads): every pass is counted."""
    g, o, info = T.build_pair("random-spheres")
    h, _ = harness("random-spheres")
    cam = T.CAMERAS["random-spheres"]
    rays = o.record_path_rays(cam, o.params(160, 120, 4, 50, background=info.background, seed=3, iterative=True),
                              support.random_xys(160, 120, 4, 6000, seed=1), 60000)
    rays = np.resize(rays, (700001, 7))
    _assert_query_counts(g, h, rays, 0, False)
