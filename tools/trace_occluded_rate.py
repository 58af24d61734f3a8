"""Rays per second of the closest-hit query against the occlusion (any-hit) query on the same rays:
shim_trace_closest_device (id and t) against shim_trace_occluded_device (one byte per ray), for C1, C2, C4 and C5.

Two workloads per configuration, both tiled to 2^24 rays:
  * path rays, t in [0.001, inf): about 2^20 camera and bounce rays of random samples recorded with the CPU oracle's
    integrator; most of them hit something;
  * segments between two of those rays' hit points a and b (origin a, direction b - a, t in [1e-3, 1 - 1e-3]), the
    visibility idiom of the header; both answers occur.
Both queries run on the same device buffers, timed with CUDA events after a warm-up, several repetitions each,
alternating, with a 512 MB write between timed launches so that neither finds the rays or the scene in L2 from the
launch before.  One untimed counted call of each query (the exact-node walk) gives node visits and primitive tests per
ray.  Prints one JSON line (rays/s of both queries and their ratio, the occluded fraction, the counts, whether the
answers agree, the GPU's name and power limit read in the same run); ``--out PATH`` writes it there too.  No target is
asserted.

    python tools/trace_occluded_rate.py [--configs C1,C2,C4,C5] [--rays 1048576] [--tile 16777216] [--reps 5] [--out PATH]
"""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests"), str(ROOT / "tools")]
from raytracinginoneweekendinrust_b200 import api, scenes  # noqa: E402
from trace_hit_rate import gpu_identity  # noqa: E402

SEG_T = (1e-3, 1.0 - 1e-3)


def segments(points, n, seed):
    """n segments between random pairs of the points (pairs closer than 1e-2 dropped)."""
    rs = np.random.RandomState(seed)
    a, b = rs.randint(0, len(points), n), rs.randint(0, len(points), n)
    d = points[b] - points[a]
    keep = np.linalg.norm(d, axis=1) > 1e-2
    seg = np.empty((keep.sum(), 7), np.float32)
    seg[:, 0:3], seg[:, 3:6], seg[:, 6] = points[a[keep]], d[keep], rs.uniform(0, 1, keep.sum())
    return seg


def measure(g, base, t_min, t_max, tile, reps, flush):
    import torch
    rays = np.resize(base, (tile, 7))
    n = len(rays)
    d_rays = torch.from_numpy(rays).cuda()
    d_prim = torch.empty(n, dtype=torch.int32, device="cuda")
    d_t = torch.empty(n, dtype=torch.float32, device="cuda")
    d_occ = torch.empty(n, dtype=torch.uint8, device="cuda")
    lib = g.lib
    stream = torch.cuda.current_stream()

    def closest():
        rc = lib.shim_trace_closest_device(g.ptr, d_rays.data_ptr(), n, t_min, t_max, 0, d_prim.data_ptr(), d_t.data_ptr(),
                                           stream.cuda_stream)
        assert rc == 0, lib.shim_last_error()

    def occluded():
        g.trace_occluded_device(d_rays.data_ptr(), n, d_occ.data_ptr(), t_min, t_max, seed=0, stream=stream.cuda_stream)

    def timed(fn):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    closest(); occluded(); torch.cuda.synchronize()          # warm-up: module load, scene upload
    tc, to = [], []
    for _ in range(reps):
        tc.append(timed(closest))
        to.append(timed(occluded))
    # the answers agree bit for bit (tests/test_occlusion.py): checked here on the timed rays
    same = bool(torch.equal(d_occ.bool(), d_prim >= 0))
    occ_frac = float(d_occ.float().mean().item())
    del d_rays, d_prim, d_t, d_occ
    torch.cuda.empty_cache()
    # one untimed counted call of each (exact nodes)
    _, _, cc = g.trace_closest(rays, t_min, t_max, seed=0, counters=True)
    _, co = g.trace_occluded(rays, t_min, t_max, seed=0, counters=True)
    mc, mo = float(np.median(tc)), float(np.median(to))
    return {
        "t_min": t_min, "t_max": t_max, "rays": n, "recorded_rays": int(len(base)), "occluded_fraction": occ_frac,
        "trace_closest_ms": [round(x, 3) for x in tc], "trace_occluded_ms": [round(x, 3) for x in to],
        "trace_closest_rays_per_s": n / (mc * 1e-3), "trace_occluded_rays_per_s": n / (mo * 1e-3),
        "occluded_over_closest_rate": mc / mo, "same_answers": same,
        "closest_nodes_per_ray": int(cc[1]) / n, "occluded_nodes_per_ray": int(co[1]) / n,
        "closest_prims_per_ray": int(cc[2]) / n, "occluded_prims_per_ray": int(co[2]) / n,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C1,C2,C4,C5")
    ap.add_argument("--rays", type=int, default=1 << 20)
    ap.add_argument("--tile", type=int, default=1 << 24)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import support
    assert torch.cuda.is_available(), "needs a CUDA device"
    name, power = gpu_identity()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    result = {"tool": "trace_occluded_rate", "gpu": name, "power_limit": power, "rays": a.tile, "reps": a.reps,
              "l2": "512 MB written between timed launches", "counts": "one untimed counted call each, exact-node walk",
              "configs": {}}
    for key in a.configs.split(","):
        cfg = scenes.configs()[key]
        o = support.OracleScene()
        info = scenes.build(o, cfg.scene, seed=1, **cfg.scene_kwargs)
        po = o.params(cfg.width, cfg.height, cfg.spp, 50, background=info.background, seed=7, iterative=True)
        xys = support.random_xys(cfg.width, cfg.height, cfg.spp, a.rays // 2, seed=3)
        base = o.record_path_rays(cfg.camera, po, xys, a.rays)
        del o
        g = api.Scene()
        scenes.build(g, cfg.scene, seed=1, **cfg.scene_kwargs)
        rec = g.trace_hit(base, seed=0)
        seg = segments(rec["point"][rec["hittable"] >= 0], len(base), seed=5)
        result["configs"][key] = {
            "scene": cfg.scene,
            "path_rays": measure(g, base, 0.001, float("inf"), a.tile, a.reps, flush),
            "segments": measure(g, seg, *SEG_T, a.tile, a.reps, flush),
        }
        del g
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
