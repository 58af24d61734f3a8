#!/usr/bin/env python
"""bench.py — Mrays/s of the path-tracing hot path on N B200s (one process per GPU).

A *step* is one full render of the workload (BASELINE.json config C1 by default: Book-1
random-spheres, 1200x800, 10 spp, depth 50) — every sample's camera ray generation, BVH
traversal + intersection and scatter/shade, i.e. everything under Renderer::render
(reference src/renderer.rs:42-105) except the PPM write.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C1] [--impl reference] [--dump-outputs DIR]

The one JSON line carries, next to the headline (`value`, C1 device-timed):
  parity    the framebuffer of the TIMED configuration against the CPU oracle on the same Philox stream
  roofline  the dominant kernel against its binding ceiling (instruction issue) with the HBM fraction beside it
  configs   BASELINE.json's other configurations (C2..C5 and their variants) at a bounded sample count each:
            Mrays/s, samples/s, end to end, roofline, the CPU arm timed beside it
  strong    (N > 1) ONE fixed image sharded over the N ranks, one NCCL reduce, against rank 0 rendering it alone

N > 1 (launched by torch.distributed.run): sample-range sharding.  `value` is weak scaling — every rank
renders `spp_per_gpu` samples per pixel of its own absolute sample range over the full image (the image
then has N x spp_per_gpu samples; `config.spp` says so), one framebuffer reduce over NCCL at the end; no
collective inside the wavefront loop.

--dump-outputs DIR writes the last timed step's output as .npy files (see dump_outputs) so that two builds can be
compared output for output: the inputs depend only on the arguments.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
# the benchmark leaves the tree as build() left it (it may be read-only): it imports modules build() does not
# (scenes, meshes, distributed), and their bytecode caches would otherwise be written next to the sources
sys.dont_write_bytecode = True

METRIC = "Mrays/s"
DUMP_BYTES = 64 << 20     # --dump-outputs: at most this much in all
DUMP_SAMPLE_PIXELS = 1 << 21   # 40 MB with their indices


# --------------------------------------------------------------------------------------------
def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


class ClockSampler:
    """SM clock + throttle reasons sampled during the timed region: NVML in a thread (every 2 ms; a Book-1 timed
    region lasts ~60 ms), nvidia-smi -lms as the fallback."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.nvml = None
        self.samples = []      # (sm MHz, max MHz, reasons bitmask)
        self._stop = threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(visible.split(",")[self.gpu]) if visible and visible.split(",")[self.gpu].strip().isdigit() else self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml

            def loop():
                while not self._stop.is_set():
                    try:
                        self.samples.append((pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM), mx,
                                             pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)))
                    except Exception:
                        break
                    time.sleep(0.002)

            self.t = threading.Thread(target=loop, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def _stop_nvml(self) -> dict:
        self._stop.set()
        self.t.join(timeout=1)
        n = self.nvml
        bits = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": n.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksEventReasonSwPowerCap}
        reasons = sorted(k for k, b in bits.items() if any(s[2] & b for s in self.samples))
        sm = [s[0] for s in self.samples]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(self.samples[0][1]) if sm else None,
                "reasons": reasons, "samples": len(sm), "source": "nvml"}

    def stop(self) -> dict:
        if self.nvml is not None:
            try:
                return self._stop_nvml()
            except Exception as e:   # fall through to whatever nvidia-smi gathered (nothing, if it was not started)
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"nvml: {e}"]}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload(args):
    from raytracinginoneweekendinrust_b200 import scenes
    cfg = scenes.configs()[args.config]
    spp = args.spp if args.spp > 0 else cfg.spp
    W = args.width if args.width > 0 else cfg.width
    H = args.height if args.height > 0 else cfg.height
    return cfg, W, H, spp


def scene_kwargs(cfg, args, extra=None):
    kw = dict(cfg.scene_kwargs)
    if extra:
        kw.update(extra)
    if args.tris > 0 and cfg.scene in ("bunny", "gargoyle", "igea-hrpp"):
        kw["n_tris"] = args.tris
    return kw


def config_dict(cfg, W, H, spp_per_gpu, n_gpus):
    """Only what names the workload (identical in both arms): under weak scaling every GPU renders spp_per_gpu samples
    per pixel of its own sample range, so the image has n_gpus x spp_per_gpu samples."""
    return {"workload": f"{cfg.key} {cfg.scene} {W}x{H} {spp_per_gpu}spp depth{cfg.max_depth}", "scene": cfg.scene, "width": W, "height": H,
            "spp": spp_per_gpu * n_gpus, "spp_per_gpu": spp_per_gpu, "max_depth": cfg.max_depth, "scene_seed": 1, "tile": "8x8",
            "l2": "256 MiB buffer written between timed steps (L2 flush)"}


# BASELINE.json's other configurations and their variants: (label, config key, scene kwargs, time the CPU arm too)
EXTRA = [
    ("C2", "C2", {}, True),
    ("C3", "C3", {"material": "lambertian"}, True),
    ("C3-dielectric", "C3", {"material": "dielectric"}, False),
    ("C3-metal", "C3", {"material": "metal"}, False),
    ("C4", "C4", {"predictors": False}, True),
    ("C4-hrpp", "C4", {"predictors": True}, False),
    ("C5", "C5", {"predictor": False}, True),
    ("C5-hrpp", "C5", {"predictor": True}, True),
]
# SURVEY.md §8d instruction budget: 30 per box test (60 per 64-byte node = both child boxes), per primitive test by
# the scene's dominant primitive (f64 sphere 2 x 45, triangle 45, Cornell's rect / six-rect cube / medium mix 60),
# 150 for shading when the dominant kernel shades too (wf_trace_solo)
PRIM_BUDGET = {"random-spheres": 90, "cornell-smoke": 60, "bunny": 45, "igea-hrpp": 45, "gargoyle": 45, "showcase": 90}
PRIM_BYTES = {"random-spheres": 32, "cornell-smoke": 32, "showcase": 32}


# -------------------------------------------------------------------------------------------- CPU arm
def run_cpu(cfg, W, H, spp, kw, steps, warmup, budget_s, threads=0):
    """The reference's path on the host cores: the C++ restatement in oracle/ in reference mode
    (recursive both-children traversal, per-node divides, f64 spheres, recursion, 8x8 tiles pulled by
    one thread per logical core), xorshift RNG standing in for thread_rng.  Each step renders a bounded
    sample of the workload (fewer spp; throughput does not depend on spp) sized from a 1-spp calibration
    so that warmup + steps stay within ``budget_s`` seconds."""
    sys.path.insert(0, str(ROOT / "tests"))
    import support
    from raytracinginoneweekendinrust_b200 import scenes
    o = support.OracleScene()
    info = scenes.build(o, cfg.scene, seed=1, **kw)

    # bounded sample: configurations above a megapixel (C3, C5) are timed on a window-preserving reduced image (same camera,
    # same scene, W/k x H/k pixels; rays per sample and the per-ray cost do not depend on the pixel count)
    k = 1
    while (W // k) * (H // k) > 1_000_000:
        k += 1
    W, H = W // k, H // k

    def params(n_spp):
        return o.params(W, H, n_spp, cfg.max_depth, background=info.background, seed=0, rng_fast=True, iterative=False,
                        threads=threads, use_predictors=info.predictors)

    _, cal = o.render(cfg.camera, params(1))
    per_spp = max(cal.seconds, 1e-4)
    cpu_spp = int(max(1, min(spp, budget_s / max(1, steps + warmup) / per_spp)))
    times, best = [], None
    for i in range(warmup + steps):
        _, st = o.render(cfg.camera, params(cpu_spp))
        if i >= warmup:
            times.append(st.seconds)
            best = st
    sec = float(np.mean(times))
    o.close()
    return {"mrays": best.rays / sec / 1e6, "samples_per_s": best.samples / sec, "seconds": sec, "threads": int(best.threads),
            "rays": int(best.rays), "sample": f"{cfg.scene} {W}x{H} at {cpu_spp} spp (of {spp}), depth {cfg.max_depth}, "
                                              f"{steps} timed render(s) after {warmup} warm-up" + (", predictors on" if info.predictors else ""),
            "nodes_per_ray": best.node_visits / max(1, best.rays), "prims_per_ray": best.prim_tests / max(1, best.rays)}


def cpu_entry(c):
    return {"value": c["mrays"], "unit": "Mrays/s", "cores": c["threads"], "kind": "port", "sample": c["sample"],
            "samples_per_s": c["samples_per_s"], "ref_nodes_per_ray": c["nodes_per_ray"], "ref_prims_per_ray": c["prims_per_ray"]}


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    result_out = _claim_stdout()
    cfg, W, H, spp = workload(args)
    r = run_cpu(cfg, W, H, spp, scene_kwargs(cfg, args), args.steps, args.warmup, budget_s=120.0)
    line = {"impl": "reference", "metric": METRIC, "value": r["mrays"], "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": r["seconds"] * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 (+f64 sphere quadratic)", "data": "synthetic",
            "config": config_dict(cfg, W, H, spp, args.gpus),
            "samples_per_s": r["samples_per_s"],
            "cpu_baseline": {"value": r["mrays"], "unit": "Mrays/s", "cores": r["threads"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": r["mrays"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "reference is Rust (no rustc here): C++ restatement in oracle/ run in reference mode on the host cores"}
    print(json.dumps(line), file=result_out, flush=True)


# -------------------------------------------------------------------------------------------- GPU arm
def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries under us write there too (NCCL prints its version banner to
    stdout): keep a private handle on the real stdout for the result line and point fd 1 at stderr for everything else."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def dump_outputs(out_dir, image, counts):
    """What the timed path returned in its last step: ``framebuffer.npy``, the (H, W, 3) float32 raw per-pixel sums
    (RENDER_RAW_SUM, reduced over the ranks), and ``counts.npy``, float64 [rays, samples] of that step over all ranks.
    An image larger than DUMP_BYTES is written as a fixed, seeded sample of its pixels instead:
    ``framebuffer_sample.npy`` (n, 3) and ``framebuffer_sample_index.npy``, their row-major pixel indices (float64).
    The counts repeat exactly from run to run; the sums only to a few float32 ulps, since the samples of a pixel are
    added in the order their paths finish."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "counts.npy", np.asarray(counts, np.float64))
    if image.nbytes + 4096 <= DUMP_BYTES:     # (room for the .npy headers and counts.npy)
        np.save(out / "framebuffer.npy", image)
        return
    n_px = image.shape[0] * image.shape[1]
    idx = np.sort(np.random.default_rng(0).choice(n_px, min(n_px, DUMP_SAMPLE_PIXELS), replace=False))
    np.save(out / "framebuffer_sample.npy", image.reshape(n_px, 3)[idx])
    np.save(out / "framebuffer_sample_index.npy", idx.astype(np.float64))


def load_ncu():
    """ncu figures per config (thread instructions per ray, active lanes, issue utilisation, DRAM bytes) measured once
    per kernel change under gpurun and committed under profiles/ (tools/ncu_summary.py writes the file)."""
    p = ROOT / "profiles" / "r02_ncu.json"
    return json.loads(p.read_text()) if p.exists() else {}


def roofline_entry(scene_name, kernel, fused, st_cnt, prof_stats, clocks, ncu):
    """Roofline of the dominant (closest-hit) kernel from the event-timed profile pass: the binding ceiling is
    instruction issue (SURVEY.md §8d), HBM is reported beside it."""
    peak_hbm, peak_src, sm_max = load_peaks()
    nodes_per_ray = st_cnt.node_visits / max(1, st_cnt.rays)
    prims_per_ray = st_cnt.prim_tests / max(1, st_cnt.rays)
    ext_ms = sum(s.extend_ms for s in prof_stats)
    ext_launch = sum(s.extend_launches for s in prof_stats)
    rays = sum(s.rays for s in prof_stats)
    prof_ms = sum(s.device_ms for s in prof_stats)
    if ext_ms <= 0 or rays <= 0:
        return None
    hbm_bytes_per_ray = 128.0   # SURVEY §8d B_state: the ray record in, ray + hit record out, amortised accumulate traffic
    onchip_bytes_per_ray = nodes_per_ray * 64 + prims_per_ray * PRIM_BYTES.get(scene_name, 48)
    sm_clk = (clocks.get("sm_mhz") or sm_max) * 1e6
    budget = nodes_per_ray * 2 * 30 + prims_per_ray * PRIM_BUDGET.get(scene_name, 45) + (150 if fused else 0)
    issue_peak = 148 * 128 * sm_clk / budget / 1e6          # Mrays/s at 32 of 32 lanes and every issue slot used
    achieved = rays / (ext_ms / 1e3) / 1e6                   # Mrays/s inside the kernel
    hbm_achieved = hbm_bytes_per_ray * rays / (ext_ms / 1e3) / 1e9
    r = {"bound": "issue", "kernel": kernel, "achieved": achieved, "peak": issue_peak, "unit": "Mrays/s", "frac": achieved / issue_peak,
         "peak_definition": "148 SMs x 4 schedulers x 32 lanes x SM clock / budgeted instructions per ray (SURVEY.md §8d: 60 per node, "
                            f"{PRIM_BUDGET.get(scene_name, 45)} per primitive test" + (", 150 shading" if fused else "") + ")",
         "budget_inst_per_ray": budget, "sm_mhz": sm_clk / 1e6, "nodes_per_ray": nodes_per_ray, "prims_per_ray": prims_per_ray,
         "kernel_ms_per_step": ext_ms / max(1, len(prof_stats)), "kernel_share_of_step": ext_ms / prof_ms if prof_ms else None,
         "kernel_launches_per_step": ext_launch / max(1, len(prof_stats)),
         "hbm": {"achieved_gbs": hbm_achieved, "peak_gbs": peak_hbm, "frac": hbm_achieved / peak_hbm, "peak_source": peak_src,
                 "algorithmic_bytes_per_ray": hbm_bytes_per_ray, "algorithmic_bytes_per_step": hbm_bytes_per_ray * rays / max(1, len(prof_stats))},
         "onchip": {"bytes_per_ray": onchip_bytes_per_ray, "achieved_gbs": onchip_bytes_per_ray * rays / (ext_ms / 1e3) / 1e9,
                    "level": "shared memory (TMA-staged scene image)" if fused or scene_name in ("cornell-smoke",) else "L1/L2"},
         "measured_on": f"{len(prof_stats)} extra step(s) of the same workload right after the timed ones, CUDA events around every launch "
                        "of the kernel on its stream (timed steps carry no per-kernel events)"}
    n = ncu.get(kernel)
    r["traffic"] = None
    if n:
        # like for like: DRAM bytes and algorithmic bytes of the SAME captured launches
        r["traffic"] = n.get("dram_bytes_per_launch")
        r["ncu"] = n
        if n.get("thread_inst_per_ray"):
            r["measured_inst_per_ray"] = n["thread_inst_per_ray"]
            r["frac_vs_measured_inst"] = achieved / (148 * 128 * sm_clk / n["thread_inst_per_ray"] / 1e6)
    return r


def measure_extra(label, key, kw, with_cpu, args, api, capi, scenes, torch, dev, stream, flush, clocks, ncu):
    """One of BASELINE.json's other configurations at a bounded sample count: device-timed steps, end to end through
    the host-buffer C ABI call, roofline of its closest-hit kernel, CPU arm beside it."""
    cfg = scenes.configs()[key]
    W, H = cfg.width, cfg.height
    spp = int(max(1, min(cfg.spp, args.extra_samples // (W * H))))
    kwargs = scene_kwargs(cfg, args, kw)
    t0 = time.perf_counter()
    scene = api.Scene()
    info = scenes.build(scene, cfg.scene, seed=1, **kwargs)
    build_s = time.perf_counter() - t0
    base = capi.RENDER_RAW_SUM | (capi.RENDER_PREDICTORS if info.predictors else 0)
    p = api.make_params(W, H, spp, cfg.max_depth, background=info.background, seed=0, flags=base)
    fb = torch.empty((H, W, 3), dtype=torch.float32, device=dev)
    for _ in range(2):
        scene.render_device(cfg.camera, p, fb.data_ptr(), stream.cuda_stream)
        flush.zero_()
    ev, stats = [], []
    for _ in range(args.extra_steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        stats.append(scene.render_device(cfg.camera, p, fb.data_ptr(), stream.cuda_stream))
        b.record(stream)
        flush.zero_()
        ev.append((a, b))
    torch.cuda.synchronize(dev)
    ms = sum(a.elapsed_time(b) for a, b in ev)
    rays = sum(s.rays for s in stats)
    out = {"workload": f"{key} {cfg.scene} {W}x{H} {spp}spp (of {cfg.spp}) depth{cfg.max_depth}", "scene_args": kwargs, "notes": info.notes,
           "value": rays / ms / 1e3, "unit": "Mrays/s", "samples_per_s": sum(s.samples for s in stats) / (ms / 1e3),
           "ms_per_step": ms / len(ev), "steps": len(ev), "rays_per_sample": rays / max(1, sum(s.samples for s in stats)),
           "iterations_per_step": stats[-1].iterations, "gpu_launches_per_step": int(stats[-1].kernel_launches),
           "scene_device_bytes": scene.device_bytes(), "pool_bytes": int(stats[-1].pool_bytes), "host_scene_build_s": build_s}
    kernel = capi.Stats.EXTEND_KERNELS.get(int(stats[-1].extend_variant), "wf_extend")   # (wf_bvh1_walk: timed with wf_bvh1_list and wf_bvh1_finish)
    if info.predictors:
        st = stats[-1]
        tot = st.hrpp_true_positive + st.hrpp_false_positive + st.hrpp_no_prediction
        out["hrpp"] = {"true_positive": st.hrpp_true_positive / max(1, tot), "false_positive": st.hrpp_false_positive / max(1, tot),
                       "no_prediction": st.hrpp_no_prediction / max(1, tot), "lookups": int(tot),
                       "note": "predictions return the first hit found in a predicted leaf (bvh.rs:145-156): the image is approximate by design",
                       "verdict": "measured for parity with Bvh::with_predictor, not a speed feature: predictions land only for camera rays of "
                                  "later samples of a pixel (diffuse bounce rays never repeat a 48-bit key), and a table probe plus the "
                                  "false-positive re-walks cost more than the ~10 node visits of a SAH walk - compare `value` with the "
                                  "predictor-off entry of the same config (DESIGN.md 5b)"}
        kernel = "wf_extend<HRPP>"
    # roofline: node / primitive counters from a 1-spp counting render (predictor off: the counters need the plain walk)
    if not info.predictors:
        pc = api.make_params(W, H, 1, cfg.max_depth, background=info.background, seed=0, flags=capi.RENDER_RAW_SUM | capi.RENDER_COUNT_NODES)
        st_cnt = scene.render_device(cfg.camera, pc, fb.data_ptr(), stream.cuda_stream)
        pp = api.make_params(W, H, spp, cfg.max_depth, background=info.background, seed=0, flags=base | capi.RENDER_PROFILE)
        flush.zero_()
        prof = [scene.render_device(cfg.camera, pp, fb.data_ptr(), stream.cuda_stream)]
        out["roofline"] = roofline_entry(cfg.scene, kernel, int(stats[-1].extend_variant) == 4, st_cnt, prof, clocks, ncu.get(label, {}))
    # end to end: commit + render into a page-locked host framebuffer
    hfb = api.HostFramebuffer(H, W)
    e2e = []
    for k in range(4):
        s2 = api.Scene()
        scenes.SCENES[cfg.scene](s2, seed=1, **kwargs)       # host-side recording (untimed, like Bvh::new in the reference)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        s2.commit()
        _, st2 = s2.render(cfg.camera, api.make_params(W, H, spp, cfg.max_depth, background=info.background, seed=0, flags=base), out=hfb.array)
        dt = time.perf_counter() - t0
        if os.environ.get("BENCH_DEBUG"):
            print(f"{label} e2e step {k}: {1e3 * dt:.2f} ms (device {st2.device_ms:.2f} ms, {st2.iterations} iterations, pool {st2.pool_paths})", file=sys.stderr)
        if k > 0:
            e2e.append((dt, st2.rays))
        s2.close()
    hfb.close()
    e2e.sort()
    dt_med, rays_med = e2e[len(e2e) // 2]   # median of the three calls after the warm-up one (a host hiccup of tens of ms is common next to the CPU legs)
    out["e2e"] = {"value": rays_med / dt_med / 1e6, "unit": "Mrays/s", "ms_per_step": 1e3 * dt_med, "calls": len(e2e), "statistic": "median",
                  "h2d_bytes_per_step": scene.device_bytes(), "d2h_bytes_per_step": W * H * 12}
    scene.close()
    del fb
    if with_cpu and not args.no_cpu:
        out["cpu_baseline"] = cpu_entry(run_cpu(cfg, W, H, spp, kwargs, 1, 0, budget_s=args.extra_cpu_s))
        out["speedup_vs_cpu"] = {"device": out["value"] / out["cpu_baseline"]["value"], "e2e": out["e2e"]["value"] / out["cpu_baseline"]["value"]}
    return out


def main_gpu(args):
    result_out = _claim_stdout()
    import torch
    import torch.distributed as dist
    from raytracinginoneweekendinrust_b200 import api, capi, distributed, scenes

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this backend has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    cfg, W, H, spp = workload(args)
    kwargs = scene_kwargs(cfg, args)
    scene = api.Scene()
    info = scenes.build(scene, cfg.scene, seed=1, **kwargs)
    base_flags = capi.RENDER_RAW_SUM | (capi.RENDER_PREDICTORS if info.predictors else 0)
    total_spp = spp * world
    # weak scaling: rank r renders absolute samples [r*spp, (r+1)*spp) of a total_spp-sample image
    assert distributed.shard_samples(total_spp, rank, world) == (rank * spp, spp)
    params = api.make_params(W, H, total_spp, cfg.max_depth, background=info.background, seed=0, sample_begin=rank * spp,
                             sample_count=spp, flags=base_flags, pool_paths=args.pool)   # no per-kernel events in timed steps (~10 % of a step)
    prof_params = api.make_params(W, H, total_spp, cfg.max_depth, background=info.background, seed=0, sample_begin=rank * spp,
                                  sample_count=spp, flags=base_flags | capi.RENDER_PROFILE, pool_paths=args.pool)
    fb = torch.empty((H, W, 3), dtype=torch.float32, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream(dev)

    def step(prm=None):
        st = scene.render_device(cfg.camera, prm or params, fb.data_ptr(), stream.cuda_stream)
        if world > 1:
            dist.reduce(fb, dst=0, op=dist.ReduceOp.SUM)   # the one framebuffer sum over NVLink
        return st

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step()
        flush.zero_()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    stats = []
    wall0 = time.perf_counter()
    for k in range(args.steps):
        ev[k][0].record(stream)
        stats.append(step())
        ev[k][1].record(stream)
        if k == args.steps - 1:
            image_sum = fb.clone()   # the timed configuration's own framebuffer (raw sums; on rank 0 the reduced ones), for the parity check
        flush.zero_()  # L2 flush between timed steps (outside the event pair)
    barrier()
    wall = time.perf_counter() - wall0
    if args.dump_outputs:
        counts = torch.tensor([float(stats[-1].rays), float(stats[-1].samples)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(counts, op=dist.ReduceOp.SUM)
        if rank == 0:
            dump_outputs(args.dump_outputs, image_sum.cpu().numpy(), counts.cpu().numpy())
    # roofline pass: the same step again with CUDA events around every launch of the closest-hit kernel (on its stream)
    prof_stats = []
    for _ in range(args.profile_steps):
        flush.zero_()
        prof_stats.append(step(prof_params))
    barrier()
    clocks = sampler.stop() if rank == 0 else {}
    ms = [a.elapsed_time(b) for a, b in ev]
    tot_ms = torch.tensor([sum(ms)], dtype=torch.float64, device=dev)
    rays = torch.tensor([float(sum(s.rays for s in stats))], dtype=torch.float64, device=dev)
    samples = torch.tensor([float(sum(s.samples for s in stats))], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(rays, op=dist.ReduceOp.SUM)
        dist.all_reduce(samples, op=dist.ReduceOp.SUM)
    tot_s = float(tot_ms.item()) / 1e3
    value = float(rays.item()) / tot_s / 1e6
    samples_per_s = float(samples.item()) / tot_s

    # ---- e2e: the C-ABI call with HOST buffers.  One rank: shim_commit (flatten + scene H2D) + shim_render into a page-locked
    # host framebuffer (D2H).  N ranks: commit + render of the rank's shard + the NCCL framebuffer sum + rank 0's D2H of the image.
    e2e_ms, h2d, d2h = [], 0, W * H * 3 * 4
    e2e_rays = 0
    E2E_WARM = 4
    pinned_fb = None if args.pageable_fb else api.HostFramebuffer(H, W)
    host_fb = np.zeros((H, W, 3), np.float32) if pinned_fb is None else pinned_fb.array
    host_t = torch.from_numpy(host_fb) if world > 1 else None
    for k in range(args.e2e_steps + E2E_WARM if args.e2e_steps > 0 else 0):
        s2 = api.Scene()
        scenes.SCENES[cfg.scene](s2, seed=1, **kwargs)  # host-side recording (untimed: Bvh::new is outside render in the reference too)
        barrier()
        t0 = time.perf_counter()
        s2.commit()
        tc = time.perf_counter()
        if world == 1:
            _, st2 = s2.render(cfg.camera, params, out=host_fb)
        else:
            st2 = s2.render_device(cfg.camera, params, fb.data_ptr(), stream.cuda_stream)
            dist.reduce(fb, dst=0, op=dist.ReduceOp.SUM)
            if rank == 0:
                host_t.copy_(fb, non_blocking=True)
            torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        if os.environ.get("BENCH_DEBUG"):
            print(f"e2e step {k}: commit {1e3 * (tc - t0):.2f} ms, render {1e3 * (time.perf_counter() - tc):.2f} ms "
                  f"(device {st2.device_ms:.2f} ms, {st2.iterations} iterations)", file=sys.stderr)
        if k >= E2E_WARM:  # the first ones warm the pinned staging buffer / allocator
            e2e_ms.append(dt * 1e3)
            e2e_rays += st2.rays
        h2d = s2.device_bytes()   # the scene blob; the tile-ordered pixel table is cached on the device after the first render
        s2.close()
    e2e_t = torch.tensor([sum(e2e_ms)], dtype=torch.float64, device=dev)
    e2e_r = torch.tensor([float(e2e_rays)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_r, op=dist.ReduceOp.SUM)
    e2e_value = float(e2e_r.item()) / (float(e2e_t.item()) / 1e3) / 1e6 if e2e_ms else None

    # ---- strong scaling (N > 1): ONE fixed image (strong_spp samples per pixel) sharded over the ranks by sample range,
    # one NCCL reduce; against rank 0 rendering the whole image alone.  Device-timed, max over ranks.
    strong = None
    if world > 1:
        S = args.strong_spp
        b, c = distributed.shard_samples(S, rank, world)
        ps = api.make_params(W, H, S, cfg.max_depth, background=info.background, seed=0, sample_begin=b, sample_count=c if c > 0 else -1,
                             flags=base_flags, pool_paths=args.pool)
        p1 = api.make_params(W, H, S, cfg.max_depth, background=info.background, seed=0, flags=base_flags, pool_paths=args.pool)
        for _ in range(2):
            step(ps)
        barrier()
        sev = []
        for _ in range(args.strong_steps):
            a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream); step(ps); bb.record(stream)
            flush.zero_()
            sev.append((a, bb))
        barrier()
        tN = torch.tensor([sum(a.elapsed_time(bb) for a, bb in sev) / len(sev)], dtype=torch.float64, device=dev)
        render_only = torch.tensor([0.0], dtype=torch.float64, device=dev)
        dist.all_reduce(tN, op=dist.ReduceOp.MAX)
        t1 = torch.tensor([0.0], dtype=torch.float64, device=dev)
        if rank == 0:   # the same image on one GPU (no reduce), the other ranks wait
            scene.render_device(cfg.camera, p1, fb.data_ptr(), stream.cuda_stream)
            a, bb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            st1 = scene.render_device(cfg.camera, p1, fb.data_ptr(), stream.cuda_stream)
            bb.record(stream)
            torch.cuda.synchronize(dev)
            t1[0] = a.elapsed_time(bb)
            render_only[0] = st1.rays
        barrier()
        if rank == 0:
            strong = {"workload": f"{cfg.key} {cfg.scene} {W}x{H} {S}spp depth{cfg.max_depth}: ONE image, sample ranges over {world} ranks, one NCCL reduce",
                      "ms_1gpu": float(t1.item()), f"ms_{world}gpu": float(tN.item()), "speedup": float(t1.item()) / float(tN.item()),
                      "efficiency": float(t1.item()) / float(tN.item()) / world, "value": float(render_only.item()) / float(tN.item()) / 1e3,
                      "unit": "Mrays/s", "limits": "the longest paths of the last wave (every rank pays the full bounce-12..50 endgame for 1/N of the "
                                                   "samples) and the fixed framebuffer reduce"}

    if rank == 0:
        ncu = load_ncu()
        # ---- parity of the timed configuration: its own framebuffer against the CPU oracle, same Philox stream
        parity = None
        if not args.no_parity:
            sys.path.insert(0, str(ROOT / "tests"))
            import support
            o = support.OracleScene()
            scenes.build(o, cfg.scene, seed=1, **kwargs)
            t0 = time.perf_counter()
            ref, so = o.render(cfg.camera, o.params(W, H, total_spp, cfg.max_depth, background=info.background, seed=0, use_predictors=info.predictors))
            got = (image_sum / float(total_spp)).cpu().numpy()
            diff = np.abs(got - ref)
            total_rays = int(rays.item()) // args.steps
            parity = {"against": "CPU oracle (oracle/shimmer_oracle.cpp), same seed and Philox stream, outside the timed region",
                      "image": f"{W}x{H} {total_spp}spp: the framebuffer of the last timed step (default pool, CUDA-graph loop"
                               + (f", {world} ranks reduced" if world > 1 else "") + ")",
                      "rmse": float(np.sqrt(np.mean((got - ref) ** 2))), "max_abs": float(diff.max()),
                      "outliers_gt_1e-3": int((diff.max(axis=2) > 1e-3).sum()), "pixels": W * H,
                      "rays_gpu": total_rays, "rays_oracle": int(so.rays), "rays_equal": total_rays == int(so.rays),
                      "gate": "RMSE <= 1e-3 on linear radiance", "pass": bool(np.sqrt(np.mean((got - ref) ** 2)) <= 1e-3),
                      "oracle_seconds": time.perf_counter() - t0}
            o.close()
        # ---- roofline of the dominant kernel
        st_cnt = scene.render_device(cfg.camera, api.make_params(W, H, total_spp, cfg.max_depth, background=info.background, seed=0,
                                                                sample_begin=0, sample_count=min(spp, 2),
                                                                flags=capi.RENDER_RAW_SUM | capi.RENDER_COUNT_NODES, pool_paths=args.pool),
                                     fb.data_ptr(), stream.cuda_stream)
        variant = int(prof_stats[0].extend_variant) if prof_stats else 0
        kernel = capi.Stats.EXTEND_KERNELS.get(variant, "wf_extend")
        roofline = roofline_entry(cfg.scene, kernel, variant == 4, st_cnt, prof_stats, clocks, ncu.get(cfg.key, {})) if prof_stats else None
        cpu = None
        if world == 1 and not args.no_cpu:
            cpu = cpu_entry(run_cpu(cfg, W, H, spp, kwargs, args.steps_cpu, args.warmup_cpu, budget_s=25.0))
        extra = None
        if world == 1 and not args.no_configs and args.config == "C1":
            extra = {}
            for label, key, kw, with_cpu in EXTRA:
                t0 = time.perf_counter()
                try:
                    extra[label] = measure_extra(label, key, kw, with_cpu, args, api, capi, scenes, torch, dev, stream, flush, clocks, ncu)
                    extra[label]["bench_seconds"] = time.perf_counter() - t0
                except Exception as e:  # noqa: BLE001 — one config must not take the headline line down
                    extra[label] = {"error": f"{type(e).__name__}: {e}"}
        line = {"metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": float(tot_ms.item()) / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32 (+f64 sphere quadratic)", "data": "synthetic",
                "config": config_dict(cfg, W, H, spp, world),
                "run": {"sharding": f"sample-range x{world}", "pool_paths": int(stats[-1].pool_paths), "pool_bytes": int(stats[-1].pool_bytes),
                        "scene_device_bytes": scene.device_bytes()},
                "samples_per_s": samples_per_s, "rays_per_step": float(rays.item()) / args.steps,
                "wall_s_timed_region": wall,
                "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "ms_per_step": float(e2e_t.item()) / max(1, len(e2e_ms)),
                        "what": ("shim_commit (flatten + scene H2D) + shim_render into a host framebuffer (D2H), host timer" if world == 1 else
                                 "per rank: shim_commit + render of its sample range; then the NCCL framebuffer sum and rank 0's D2H of the image; "
                                 "host timer, max over ranks") + "; scene recording incl. the SAH tree build is outside (Bvh::new is outside "
                                "Renderer::render in the reference too)",
                        "host_framebuffer": "pageable" if args.pageable_fb else "page-locked (shim_host_alloc)"},
                "gpu_launches": int(sum(s.kernel_launches for s in stats)),
                "iterations_per_step": float(np.mean([s.iterations for s in stats])),
                "parity": parity, "roofline": roofline, "cpu_baseline": cpu, "strong": strong, "configs": extra}
        print(json.dumps(line), file=result_out, flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C1")
    ap.add_argument("--spp", type=int, default=0)
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--tris", type=int, default=0)
    ap.add_argument("--pool", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=8)
    ap.add_argument("--pageable-fb", action="store_true", help="e2e: ordinary (pageable) host framebuffer instead of shim_host_alloc")
    ap.add_argument("--profile-steps", type=int, default=3)
    ap.add_argument("--steps-cpu", type=int, default=2)
    ap.add_argument("--warmup-cpu", type=int, default=1)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline only: skip BASELINE.json's other configurations")
    ap.add_argument("--extra-samples", type=float, default=1.0e8, help="samples per step of each extra configuration")
    ap.add_argument("--extra-steps", type=int, default=3)
    ap.add_argument("--extra-cpu-s", type=float, default=5.0)
    ap.add_argument("--strong-spp", type=int, default=160)
    ap.add_argument("--strong-steps", type=int, default=5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's framebuffer and ray / sample counts as .npy files under DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        main_reference(args)
    else:
        main_gpu(args)


if __name__ == "__main__":
    main()
