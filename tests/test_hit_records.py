"""Hittable::hit with the whole HitRecord (shim_trace_hit): record-level parity with the oracle.

On the CPU the product's device arithmetic (tests/hostsim: closest_hit + reconstruct_hit, as trace_hit_kernel runs
them) must give the oracle's record bit for bit, every field compared as raw bits.  With -m gpu the CUDA kernel is
compared the same way; there the device acosf / atan2f of the sphere uv and the device logf of a medium's free path
may differ from glibc by an ulp (stated per test)."""
import ctypes as C

import numpy as np
import pytest

import records_support as R
import support
import test_gpu_parity as T
from fuzz_scenes import build_random_scene, random_rays
from raytracinginoneweekendinrust_b200 import api, capi, scenes

MEDIA_SCENES = ("cornell-smoke", "showcase")


def words(rec):
    """(n, 12) uint32: every field of every record as raw bits."""
    return np.ascontiguousarray(rec).view(np.uint32).reshape(-1, 12)


def assert_records_identical(a, b, what=""):
    wa, wb = words(a), words(b)
    bad = np.nonzero((wa != wb).any(axis=1))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} of {len(wa)} records differ, first {bad[:5]}: {a[bad[:2]]} vs {b[bad[:2]]}"


class _Kinds:
    """Forwards the builder calls to a scene and remembers which hittable ids are spheres / moving spheres / media."""

    def __init__(self, s):
        self.s, self.spheres, self.media = s, set(), set()

    def __getattr__(self, name):
        return getattr(self.s, name)

    def sphere(self, *a, **k):
        i = self.s.sphere(*a, **k); self.spheres.add(i); return i

    def moving_sphere(self, *a, **k):
        i = self.s.moving_sphere(*a, **k); self.spheres.add(i); return i

    def constant_medium(self, *a, **k):
        i = self.s.constant_medium(*a, **k); self.media.add(i); return i

    def constant_medium_color(self, boundary, density, rgb):
        return self.constant_medium(boundary, density, self.s.texture_solid(*rgb))


def scene_rays(o, name, info, n_paths=1500, cap=20000, seed=4):
    """Path rays the oracle's integrator traces in the scene, then as many random rays: origins on those paths,
    directions uniform on the sphere, times in [0, 1)."""
    cam = T.CAMERAS[name]
    W, H, spp = 120, 90, 4
    po = o.params(W, H, spp, 50, background=info.background, seed=13, iterative=True)
    path = o.record_path_rays(cam, po, support.random_xys(W, H, spp, n_paths, seed=seed), cap)
    rs = np.random.RandomState(seed)
    k = min(len(path), 6000)
    rnd = np.empty((k, 7), np.float32)
    rnd[:, 0:3] = path[rs.randint(0, len(path), k), 0:3]
    d = rs.normal(size=(k, 3))
    rnd[:, 3:6] = d / np.linalg.norm(d, axis=1, keepdims=True)
    rnd[:, 6] = rs.uniform(0, 1, k)
    return np.concatenate([path, rnd])


# ------------------------------------------------------------------------------------------------ CPU (hostsim)
@pytest.mark.parametrize("reference_tree", [False, True])
@pytest.mark.parametrize("name", list(scenes.SCENES))
def test_device_records_match_oracle_bit_for_bit(name, reference_tree):
    kw = T.SMALL.get(name, {})
    o, h = R.OracleScene(), R.HostSimScene()
    info = scenes.build(o, name, seed=1, **kw)
    h.set_device_bvh(reference_tree)
    scenes.build(h, name, seed=1, **kw)
    rays = scene_rays(o, name, info)
    ref = o.trace_hit(rays, seed=13)
    dev, cnt = h.trace_hit(rays, seed=13, counters=True)
    # An exact tie between coplanar faces of two primitives (showcase's ground cubes share faces) can go to the other
    # primitive on the device walk of the recorded bvh.rs tree: same t, the other id - shim_trace_closest answers the
    # same (checked below), so it is a closest-hit tie-break, not a record difference.  Every other record is identical.
    mism = ref["hittable"] != dev["hittable"]
    tie = mism & (ref["t"].view(np.uint32) == dev["t"].view(np.uint32)) & (ref["hittable"] >= 0) & (dev["hittable"] >= 0)
    np.testing.assert_array_equal(mism, tie)
    assert tie.sum() <= (0 if name != "showcase" else max(2, len(rays) // 5000)), f"{tie.sum()} ties"
    assert_records_identical(ref[~mism], dev[~mism], name)
    assert (ref["hittable"] >= 0).sum() > len(rays) // 8
    # hittable / t are what the closest-hit query of the same walk returns, bit for bit
    p, t, cnt_closest = h.trace_closest(rays, seed=13, counters=True)
    np.testing.assert_array_equal(dev["hittable"], p)
    np.testing.assert_array_equal(dev["t"].view(np.uint32), t.view(np.uint32))
    assert list(cnt) == list(cnt_closest)


@pytest.mark.parametrize("name", ["bunny", "gargoyle", "igea-hrpp"])
def test_quantised_mesh_walk_gives_the_same_records(name):
    """A mesh among the Cornell rects is queried on its quantised nodes (what the kernel walks for such a scene)."""
    kw = T.SMALL.get(name, {})
    o, h = R.OracleScene(), R.HostSimScene()
    info = scenes.build(o, name, seed=1, **kw)
    scenes.build(h, name, seed=1, **kw)
    rays = scene_rays(o, name, info)
    ref = o.trace_hit(rays, seed=2)
    assert_records_identical(ref, h.trace_hit(rays, seed=2, quantised=True), name + " quantised")
    assert_records_identical(ref, h.trace_hit(rays, seed=2), name + " exact nodes")


@pytest.mark.parametrize("reference_tree", [False, True])
@pytest.mark.parametrize("seed", range(6))
def test_fuzz_scene_records_match_oracle(seed, reference_tree):
    o, h = R.OracleScene(), R.HostSimScene()
    build_random_scene(o, seed)
    h.set_device_bvh(reference_tree)
    build_random_scene(h, seed)
    rays = random_rays(seed, 6000)
    ref = o.trace_hit(rays, seed=seed)
    assert_records_identical(ref, h.trace_hit(rays, seed=seed), f"fuzz seed {seed}")
    assert (ref["hittable"] >= 0).sum() > 1000


def _field_scene(s):
    """One object of every kind, 6 apart along x; returns their ids and the medium's expected phase material."""
    ids = {}
    m_diffuse = s.lambertian_color(0.5, 0.5, 0.5)
    m_metal = s.material_metal(0.8, 0.8, 0.8, 0.1)
    m_glass = s.material_dielectric(1.5)
    ids["sphere"] = s.sphere((0.0, 0.0, 0.0), 1.0, m_diffuse)
    ids["moving_sphere"] = s.moving_sphere((6.0, 0.0, 0.0), (6.0, 0.5, 0.0), 0.0, 1.0, 1.0, m_metal)
    ids["xy_rect"] = s.xy_rect(11.0, 13.0, -1.0, 1.0, 0.0, m_diffuse)
    ids["xz_rect"] = s.xz_rect(17.0, 19.0, -1.0, 1.0, 0.0, m_glass)
    ids["yz_rect"] = s.yz_rect(-1.0, 1.0, -1.0, 1.0, 24.0, m_metal)
    ids["tri"] = s.tri((29.0, -1.0, -1.0), (31.0, -1.0, 0.5), (30.0, 1.0, 0.0), m_diffuse)
    ids["cube"] = s.cube((35.0, -1.0, -1.0), (37.0, 1.0, 1.0), m_glass)
    ids["rotated_cube"] = s.translate(s.rotate_y(s.cube((-1.0, -1.0, -1.0), (1.0, 1.0, 1.0), m_metal), 70.0), (42.0, 0.0, 0.0))
    ids["translated_sphere"] = s.translate(s.sphere((0.0, 0.0, 0.0), 1.0, m_glass), (48.0, 0.0, 0.0))
    phase = 3                                      # three materials so far: the medium's Isotropic takes the next id
    ids["medium"] = s.constant_medium(s.sphere((54.0, 0.0, 0.0), 1.0, m_diffuse), 2.0, s.texture_solid(0.9, 0.9, 0.9))
    after = s.material_lambertian(s.texture_solid(0.1, 0.2, 0.3))
    for k in ids:
        s.world_add(ids[k])
    s.commit()
    return ids, phase, after


def _aimed_rays(centres, per, seed):
    rs = np.random.RandomState(seed)
    out = []
    for c in centres:
        d = rs.normal(size=(per, 3))
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        org = np.asarray(c) + d * rs.uniform(2.5, 4.0, (per, 1))
        tgt = np.asarray(c) + rs.uniform(-1.0, 1.0, (per, 3))
        r = np.concatenate([org, tgt - org, rs.uniform(0, 1, (per, 1))], axis=1)
        out.append(r)
    return np.concatenate(out).astype(np.float32)


def test_every_record_field_is_covered():
    """Sphere and moving-sphere uv, rect uv, cube sides, the triangle normal, RotateY's mixed-space set_face_normal with
    front_face left as the inner hit set it, Translate's moved point and the medium record, against the oracle."""
    o, h = R.OracleScene(), R.HostSimScene()
    ids, phase, after = _field_scene(o)
    assert _field_scene(h) == (ids, phase, after)
    assert after == phase + 1
    centres = [(6.0 * i, 0.0, 0.0) for i in range(len(ids))]
    rays = _aimed_rays(centres, 3000, seed=5)
    ref = o.trace_hit(rays, seed=7)
    dev = h.trace_hit(rays, seed=7)
    assert_records_identical(ref, dev, "field scene")
    by = {k: dev[dev["hittable"] == v] for k, v in ids.items() if k not in ("rotated_cube", "translated_sphere", "medium")}
    for k in by:
        assert len(by[k]) > 200, k
    # sphere uv: sphere.rs:41-46, both in [0, 1] and spread over the sphere
    for k in ("sphere", "moving_sphere"):
        u, v = by[k]["u"], by[k]["v"]
        assert (u >= 0).all() and (u <= 1).all() and (v >= 0).all() and (v <= 1).all()
        assert u.std() > 0.1 and v.std() > 0.1, k
    for k in ("xy_rect", "xz_rect", "yz_rect"):
        u, v = by[k]["u"], by[k]["v"]
        assert (u >= 0).all() and (u <= 1).all() and u.std() > 0.1 and v.std() > 0.1, k
    # cube: all six sides answer, each with its axis normal turned against the ray
    n = by["cube"]["normal"]
    assert len({tuple(x) for x in n.tolist()}) == 6
    assert (np.abs(n).sum(axis=1) == 1).all()
    # triangle: one normal up to the sign, face-forwarded
    tn = by["tri"]["normal"]
    e1, e2 = np.float32([2.0, 0.0, 1.5]), np.float32([1.0, 2.0, 1.0])
    want = np.cross(e1, e2); want /= np.linalg.norm(want)
    assert np.allclose(np.abs(tn @ want), 1.0, atol=1e-6)
    assert set(by["tri"]["front_face"].tolist()) == {0, 1}
    # RotateY: set_face_normal with the rotated ray while front_face keeps the inner value, so the world-space normal
    # can point along the ray; the translated point lies on the rotated cube around (42, 0, 0)
    on_rc = (dev["hittable"] >= 0) & (dev["point"][:, 0] > 39.0) & (dev["point"][:, 0] < 45.0)
    assert on_rc.sum() > 200
    along = (rays[on_rc, 3:6] * dev[on_rc]["normal"]).sum(axis=1) > 0
    assert along.any() and (~along).any()
    ts = dev[(dev["point"][:, 0] > 46.5) & (dev["point"][:, 0] < 49.5) & (dev["hittable"] >= 0)]
    assert len(ts) > 200 and np.allclose(np.linalg.norm(ts["point"] - np.float32([48, 0, 0]), axis=1), 1.0, atol=1e-4)
    # medium: hittable.rs:216-231, the phase material allotted by shim_constant_medium
    med = dev[dev["hittable"] == ids["medium"]]
    assert len(med) > 100
    assert (med["normal"] == np.float32([1, 0, 0])).all() and (med["front_face"] == 1).all()
    assert (med["u"] == 0).all() and (med["v"] == 0).all() and (med["material"] == phase).all()


def test_miss_record_is_exact():
    o, h = R.OracleScene(), R.HostSimScene()
    for s in (o, h):
        scenes.build(s, "random-spheres", seed=1)
    rays = np.array([[0, 50, 0, 0, 1, 0, 0], [0, 2000, 0, 1, 0.5, 0, 0.5]], np.float32)
    for rec in (o.trace_hit(rays), h.trace_hit(rays)):
        want = np.zeros(2, capi.HIT_RECORD_DTYPE)
        want["t"] = np.inf
        want["material"] = -1
        want["hittable"] = -1
        assert_records_identical(want, rec, "miss")
    assert len(h.trace_hit(np.zeros((0, 7), np.float32))) == 0


def test_record_layout_is_the_headers():
    assert C.sizeof(capi.HitRecord) == capi.HIT_RECORD_DTYPE.itemsize == 48
    for name, _ in capi.HitRecord._fields_:
        assert getattr(capi.HitRecord, name).offset == capi.HIT_RECORD_DTYPE.fields[name][1], name
    assert [n for n, _ in capi.HitRecord._fields_] == ["point", "normal", "t", "u", "v", "front_face", "material", "hittable"]


def test_rust_sys_record_has_the_headers_fields_in_order():
    from test_rust_binding import _c_struct_fields, _rust_struct_fields
    fields = _c_struct_fields("shim_hit_record")
    assert fields == [n for n, _ in capi.HitRecord._fields_]
    assert _rust_struct_fields("shim_hit_record") == fields


def _has_cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_state_and_argument_errors_without_a_commit():
    """An uncommitted scene is a state error for both variants, a null scene an invalid argument; nothing is written."""
    s = api.Scene()
    out = np.full(1, 7, capi.HIT_RECORD_DTYPE)
    for call in (lambda: s.trace_hit(np.zeros((1, 7), np.float32)), lambda: s.trace_hit_device(0, 1, 0)):
        with pytest.raises(capi.ShimError) as e:
            call()
        assert e.value.code == -4 and "not committed" in e.value.message
    lib = capi.load_library()
    rays = np.zeros((1, 7), np.float32)
    assert lib.shim_trace_hit(None, rays.ctypes.data, 1, 0.001, np.inf, 0, out.ctypes.data_as(C.POINTER(capi.HitRecord)), None) == -1
    assert lib.shim_trace_hit_device(None, None, 1, 0.001, np.inf, 0, None, None) == -1
    assert (words(out) == words(np.full(1, 7, capi.HIT_RECORD_DTYPE))).all()


@pytest.mark.skipif(_has_cuda(), reason="needs a machine without a CUDA device")
def test_no_cpu_fallback_without_a_device():
    """Without a device the scene cannot be committed (SHIM_ERR_CUDA), so the query has nothing to run on: it reports
    the state error and leaves the output as it was instead of computing anything on the CPU."""
    s = api.Scene()
    scenes.random_spheres(s, seed=1)
    with pytest.raises(capi.ShimError) as e:
        s.commit()
    assert e.value.code == -3 and "no CPU fallback" in e.value.message
    out = np.full(4, 7, capi.HIT_RECORD_DTYPE)
    lib = capi.load_library()
    rays = np.zeros((4, 7), np.float32)
    rc = lib.shim_trace_hit(s.ptr, rays.ctypes.data, 4, 0.001, np.inf, 0, out.ctypes.data_as(C.POINTER(capi.HitRecord)), None)
    assert rc == -4
    assert (words(out) == words(np.full(4, 7, capi.HIT_RECORD_DTYPE))).all()


# ------------------------------------------------------------------------------------------------ GPU
def build_pair(name, seed=1):
    """The product scene and the oracle scene (with orc_trace_hit) of one of scenes.SCENES, at the parity tests' sizes."""
    g = api.Scene()
    info = scenes.build(g, name, seed=seed, **T.SMALL.get(name, {}))
    o = R.OracleScene()
    scenes.build(o, name, seed=seed, **T.SMALL.get(name, {}))
    return g, o, info


def _sphere_and_medium_ids(name):
    k = _Kinds(R.OracleScene())
    scenes.build(k, name, seed=1, **T.SMALL.get(name, {}))
    return k.spheres, k.media


def compare_gpu_to_oracle(rays, ref, gpu, spheres, media, allowed_id_flips):
    """Ids agree (up to the stated flips); where they agree, every field is bit-equal except the sphere uv (device
    acosf / atan2f: within 2e-6) and, for a medium hit, t and the point (device logf of the free path: t within 1e-5
    relative, the same ulp that can flip an accept; the point = origin + t * direction moves by that t difference
    times the direction, plus the rounding of the two f32 operations)."""
    mism = ref["hittable"] != gpu["hittable"]
    assert mism.sum() <= allowed_id_flips, f"{mism.sum()} hittable mismatches"
    ok = ~mism
    r, g = ref[ok], gpu[ok]
    med = np.isin(r["hittable"], list(media))
    sph = np.isin(r["hittable"], list(spheres))
    wr, wg = words(r), words(g)
    cols = {"point": slice(0, 3), "normal": slice(3, 6), "t": slice(6, 7), "u": slice(7, 8), "v": slice(8, 9), "ints": slice(9, 12)}
    for f in ("normal", "ints"):
        np.testing.assert_array_equal(wr[:, cols[f]], wg[:, cols[f]], err_msg=f)
    for f in ("point", "t"):
        np.testing.assert_array_equal(wr[~med, cols[f]], wg[~med, cols[f]], err_msg=f)
    if med.any():
        ta, tb = r["t"][med].astype(np.float64), g["t"][med].astype(np.float64)
        assert (np.abs(ta - tb) <= 1e-5 * np.abs(ta)).all(), "t"
        d = rays[ok][med, 3:6].astype(np.float64)
        pa, pb = r["point"][med].astype(np.float64), g["point"][med].astype(np.float64)
        ulps = np.spacing(np.abs(ta[:, None] * d).astype(np.float32)) + np.spacing(np.abs(pa).astype(np.float32))
        assert (np.abs(pa - pb) <= np.abs(ta - tb)[:, None] * np.abs(d) + 2 * ulps).all(), "point"
    for f in ("u", "v"):
        np.testing.assert_array_equal(wr[~sph, cols[f]], wg[~sph, cols[f]], err_msg=f)
        if sph.any():
            assert np.abs(r[f][sph] - g[f][sph]).max() <= 2e-6, f
    return int(mism.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(scenes.SCENES))
def test_gpu_records_match_oracle(name):
    g, o, info = build_pair(name)
    cam = T.CAMERAS[name]
    W, H, spp = 160, 120, 4
    po = o.params(W, H, spp, 50, background=info.background, seed=3, iterative=True)
    rays = o.record_path_rays(cam, po, support.random_xys(W, H, spp, 6000, seed=1), 60000)
    assert len(rays) > 6000
    ref = o.trace_hit(rays, seed=3)
    gpu = g.trace_hit(rays, seed=3)
    spheres, media = _sphere_and_medium_ids(name)
    # volumes draw ln(U): device logf differs from glibc by an ulp, which can flip an accept at a boundary
    allowed = 0 if name not in MEDIA_SCENES else max(2, len(rays) // 20000)
    compare_gpu_to_oracle(rays, ref, gpu, spheres, media, allowed)
    # the same answer as the closest-hit query of the same rays, bit for bit
    p, t = g.trace_closest(rays, seed=3)
    np.testing.assert_array_equal(gpu["hittable"], p)
    np.testing.assert_array_equal(gpu["t"].view(np.uint32), t.view(np.uint32))
    # counters: the counted walk, the same hits and the same counts as trace_closest's
    gpu_c, cnt = g.trace_hit(rays, seed=3, counters=True)
    _, _, cnt_closest = g.trace_closest(rays, seed=3, counters=True)
    assert list(cnt) == list(cnt_closest) and cnt[0] == len(rays)
    assert_records_identical(gpu, gpu_c, name + " counted walk")


@pytest.mark.gpu
def test_gpu_device_variant_on_a_side_stream():
    import torch
    g, o, info = build_pair("cornell-smoke")
    cam = T.CAMERAS["cornell-smoke"]
    po = o.params(96, 96, 4, 50, background=info.background, seed=9, iterative=True)
    rays = o.record_path_rays(cam, po, support.random_xys(96, 96, 4, 3000, seed=3), 30000)
    n = len(rays)
    host = g.trace_hit(rays, seed=9)
    d_rays = torch.from_numpy(rays).cuda()
    d_out = torch.full((n, 12), -7, dtype=torch.int32, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        g.trace_hit_device(d_rays.data_ptr(), n, d_out.data_ptr(), seed=9, stream=side.cuda_stream)
    side.synchronize()
    dev = d_out.cpu().numpy().view(capi.HIT_RECORD_DTYPE).reshape(-1)
    assert_records_identical(host, dev, "device variant")
    # argument rules of the device variant
    for bad in (lambda: g.trace_hit_device(d_rays.data_ptr(), n, d_out.data_ptr() + 4),          # not 16-byte aligned
                lambda: g.trace_hit_device(d_rays.data_ptr(), -1, d_out.data_ptr()),
                lambda: g.trace_hit_device(0, n, d_out.data_ptr())):
        with pytest.raises(capi.ShimError) as e:
            bad()
        assert e.value.code == -1
    g.trace_hit_device(0, 0, 0)                                                                    # n == 0: no-op
    assert len(g.trace_hit(np.zeros((0, 7), np.float32))) == 0


@pytest.mark.gpu
def test_gpu_grid_stride_batch():
    """More rays than the grid has threads (148 SMs x 2048), a count that is not a multiple of the block size:
    every record is written and right.  Rays of a scene without media repeat with the period of the tiling."""
    g, o, info = build_pair("random-spheres")
    cam = T.CAMERAS["random-spheres"]
    po = o.params(160, 120, 4, 50, background=info.background, seed=5, iterative=True)
    base = o.record_path_rays(cam, po, support.random_xys(160, 120, 4, 4000, seed=2), 40000)
    n = 700001
    assert n % 256 and n > 148 * 2048
    rays = np.resize(base, (n, 7))
    gpu = g.trace_hit(rays, seed=5)
    ref = o.trace_hit(base, seed=5)
    idx = np.arange(n) % len(base)
    spheres, media = _sphere_and_medium_ids("random-spheres")
    compare_gpu_to_oracle(rays, ref[idx], gpu, spheres, media, 0)
