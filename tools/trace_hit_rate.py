"""Rays per second of the two ray queries on the same rays: shim_trace_closest_device (id and t) against
shim_trace_hit_device (the whole HitRecord), for C1, C4 and C5.

About 2^20 path rays per configuration are recorded with the CPU oracle's integrator (camera and bounce rays of random
samples) and tiled to 2^24.  Both queries run on the same device buffers, timed with CUDA events after a warm-up,
several repetitions each, alternating, with a 512 MB write between timed launches so that neither finds the rays or
the scene in L2 from the launch before.  Prints one JSON line (rays/s of both queries and their ratio per configuration,
the GPU's name and power limit read in the same run); ``--out PATH`` writes it there too.  No target is asserted.

    python tools/trace_hit_rate.py [--configs C1,C4,C5] [--rays 1048576] [--tile 16777216] [--reps 5] [--out PATH]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]
from raytracinginoneweekendinrust_b200 import api, scenes  # noqa: E402


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or q.stderr.strip()
    except Exception as e:   # the number is still reported, marked as having no power reading
        power = f"unavailable ({e})"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C1,C4,C5")
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
    result = {"tool": "trace_hit_rate", "gpu": name, "power_limit": power, "rays": a.tile, "reps": a.reps,
              "l2": "512 MB written between timed launches", "configs": {}}
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
        rays = np.resize(base, (a.tile, 7))
        n = len(rays)
        d_rays = torch.from_numpy(rays).cuda()
        d_prim = torch.empty(n, dtype=torch.int32, device="cuda")
        d_t = torch.empty(n, dtype=torch.float32, device="cuda")
        d_rec = torch.empty((n, 12), dtype=torch.int32, device="cuda")
        lib = g.lib
        stream = torch.cuda.current_stream()

        def closest():
            rc = lib.shim_trace_closest_device(g.ptr, d_rays.data_ptr(), n, 0.001, float("inf"), 0, d_prim.data_ptr(), d_t.data_ptr(),
                                               stream.cuda_stream)
            assert rc == 0, lib.shim_last_error()

        def hit():
            g.trace_hit_device(d_rays.data_ptr(), n, d_rec.data_ptr(), seed=0, stream=stream.cuda_stream)

        def timed(fn):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1)

        closest(); hit(); torch.cuda.synchronize()          # warm-up: module load, scene upload
        tc, th = [], []
        for _ in range(a.reps):
            tc.append(timed(closest))
            th.append(timed(hit))
        # the two queries agree on what was hit (bit for bit, tests/test_hit_records.py): checked here on the timed rays
        rec = d_rec.cpu().numpy().view(np.int32)
        same = bool(np.array_equal(rec[:, 11], d_prim.cpu().numpy()) and
                    np.array_equal(rec[:, 6], d_t.cpu().numpy().view(np.int32)))
        mc, mh = float(np.median(tc)), float(np.median(th))
        result["configs"][key] = {
            "scene": cfg.scene, "recorded_rays": int(len(base)), "hit_fraction": float((d_prim >= 0).float().mean().item()),
            "trace_closest_ms": [round(x, 3) for x in tc], "trace_hit_ms": [round(x, 3) for x in th],
            "trace_closest_rays_per_s": n / (mc * 1e-3), "trace_hit_rays_per_s": n / (mh * 1e-3),
            "hit_over_closest_rate": mc / mh, "same_hits": same,
        }
        del d_rays, d_prim, d_t, d_rec, g
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
