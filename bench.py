#!/usr/bin/env python
"""bench.py -- particle-steps/s of the SPHSystem::step() hot path on a synthetic dam-break.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload dfsph|wcsph|pbd] [--impl reference] [--dump-outputs DIR]

A "step" is one SPHSystem::step(): neighbour search + one solver step over the whole particle set.
Default workload at N=1: BASELINE.json configs[2], the configuration the north-star target is quoted on
(2M-particle DFSPH dam-break, dt=0.004, exactly 4 divergence + 4 density iterations).  --workload wcsph /
pbd select configs[1] / configs[3] on the same 2M scene.  N>1: x-slab decomposition, 2M particles per GPU
(weak scaling; N=8 is BASELINE configs[4], the 16M scene), see cpp-fluid-particles_b200/slabs.py.

Printed JSON (one line, rank 0):
  value       whole-job particle-steps/s, state resident in HBM, timed on the device with CUDA events over
              exactly K steps (barrier + synchronize on both sides, max over ranks)
  e2e         the same metric through the reference-facing C++ class API (SPHSystem via the sph_app facade)
              with HOST buffers: every step takes pos+vel from pinned host memory, steps, and delivers
              pos+vel+density to pinned host memory; all copies inside the timed region, pipelined against the
              previous batch's step (sph_app_submit / sph_app_wait); the blocking variant is reported beside it
  roofline    the density kernel named by BASELINE.json's metric (for DFSPH: computeDensityAlpha's
              replacement, fused with the colour gradient and the first divergence error), timed live with
              CUDA events inside the timed region; algorithmic bytes per
              particle from SURVEY.md 8(d); peak from MEASURED_PEAKS.json; `kernels` lists every sweep timed
  cpu_baseline  the CPU restatement (oracle/, OpenMP, all host cores): one warm-up + >= 3 timed steps of the
              workload's own scene (median)
  clocks      nvidia-smi samples taken during the timed region
--impl reference: the UNMODIFIED reference CUDA sources compiled for sm_100 (oracle/_ref/libsphref.so),
driven through the very same facade source -- the "reference build" of the north star -- on the same
scene, timed as the median of per-step wall times (its own cudaEvent figure is reported beside it); if that
library is absent, the CPU restatement is timed instead (kind "port").
N>1: every line is self-checked first (slabs.parity_check: two steps against a single-GPU run of the same scene).
--dump-outputs DIR (N=1): after the timed steps, the fluid state the timed path left after its last step is written as
DIR/{pos,vel,density,pressure}.npy (float32, rows in the engine's sorted order; see dump_outputs).  The scenes are
deterministic lattices, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALG_BYTES = {  # SURVEY.md section 8(d): algorithmic HBM bytes per fluid particle per kernel invocation
    "density": 20, "density_alpha": 24, "pressure_force": 48, "viscosity": 40, "color_grad": 28, "surface": 52,
    "advect": 48, "dfsph_error": 44, "dfsph_correct": 44, "pbd_lambda": 24, "pbd_delta_pos": 32, "pbd_xsph": 40,
    "neighbor_search": 126,
    # fused sweeps: the union of what the two operators read / write, shared reads counted once
    "density_alpha+color_grad": 36,   # R pos12+mass4, W density4 alpha4 colorGrad12
    "density+color_grad": 32,         # R pos12+mass4, W density4 colorGrad12
    "viscosity+surface": 76,          # viscosity 40 + surface 52 - shared pos/mass 16
    # density/alpha + colour gradient + first divergence error: R pos12 vel12 mass4, W density4 alpha4 colorGrad12 error4 stiff4
    "density_alpha+color_grad+div_error": 56,
    "pbd_xsph+color_grad": 52,        # xsph 40 + colour gradient 28 - shared pos/mass 16
}
SCENE_OF_N = {1: "2m", 2: "4m", 4: "8m", 8: "16m"}
DUMP_FIELDS = ("pos", "vel", "density", "pressure")
DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir: str, state: dict, seed: int = 0) -> None:
    """Writes state[f] for f in DUMP_FIELDS as out_dir/<f>.npy (float32).  When all rows together would exceed
    DUMP_BYTES, every array keeps the same rows: a sample drawn with a fixed seed, in increasing row order."""
    arrays = {f: np.ascontiguousarray(state[f], np.float32) for f in DUMP_FIELDS}
    n = arrays["pos"].shape[0]
    keep = min(n, (DUMP_BYTES - 4096) // (sum(a.nbytes for a in arrays.values()) // n))   # 4096: the .npy headers
    if keep < n:
        rows = np.sort(np.random.default_rng(seed).choice(n, size=keep, replace=False))
        arrays = {f: a[rows] for f, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for f, a in arrays.items():
        np.save(os.path.join(out_dir, f + ".npy"), a)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0, period_ms: int = 100):
        self.index, self.proc, self.lines, self.period_ms = index, None, [], period_ms

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line)

    def stop(self) -> dict:
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
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def ncu_traffic(kernel_substring: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the density kernel, from the committed
    `ncu --set full` capture of this round (profiles/r02/sweeps_dfsph_2m.raw.csv); None if absent."""
    import csv
    path = os.path.join(ROOT, "profiles", "r02", "sweeps_dfsph_2m.raw.csv")
    if not os.path.exists(path):
        return None, None
    try:
        rows = list(csv.reader(open(path)))
        hdr, units = rows[0], rows[1]
        for r in rows[2:]:
            d = dict(zip(hdr, r))
            if kernel_substring in d.get("Kernel Name", ""):
                tot = 0.0
                for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(units[hdr.index(k)], 1.0)
                    tot += float(d[k].replace(",", "")) * scale
                return tot, os.path.relpath(path, ROOT)
    except (OSError, ValueError, KeyError, IndexError):
        pass                                    # a malformed capture must not take the bench line down
    return None, None


def cpu_baseline(pkg, solver: str, scene_name: str = "2m", budget_s: float = 30.0) -> dict:
    """The CPU restatement (oracle/, OpenMP) on a bounded sample of the workload: the workload's own scene when one
    step fits the budget (2M particles: ~1 s/step on a 64-core box), else the next smaller scene of the same generator.
    One un-timed warm-up step (OpenMP team start-up, page faults), then >= 3 timed steps; the median is reported."""
    from oracle import oracle as O
    cores = O.use_all_cores()
    order = ["config0", "200k", "2m"]
    names = order[: order.index(scene_name) + 1] if scene_name in order else order
    out = None
    for name in reversed(names):
        sc = pkg.scene.benchmark_scene(name, solver)
        n = sc.fluid.shape[0]
        t_ctor = time.perf_counter()
        s = O.OracleSystem(sc)        # includes step 0 (Q3)
        t_ctor = time.perf_counter() - t_ctor
        t0 = time.perf_counter(); s.step(); warm = time.perf_counter() - t0          # warm-up, not reported
        if warm * 3 > budget_s and name != names[0]:
            s.close()
            continue                  # too slow on this box: sample the next smaller scene
        times = []
        while len(times) < 3 or (sum(times) < 3.0 and len(times) < 20):
            t0 = time.perf_counter(); s.step(); times.append(time.perf_counter() - t0)
        s.close()
        dt = float(np.median(times))
        out = {"value": n / dt, "unit": "particle-steps/s", "cores": cores, "kind": "port",
               "omp": {"OMP_NUM_THREADS": os.environ.get("OMP_NUM_THREADS"), "OMP_PROC_BIND": os.environ.get("OMP_PROC_BIND"),
                       "threads_used": cores},
               "sample": f"{len(times)} timed step(s) after 1 warm-up step of the {name} {solver} dam-break ({n} fluid particles): "
                         f"median {dt*1e3:.1f} ms/step (min {min(times)*1e3:.1f}, max {max(times)*1e3:.1f}; warm-up {warm*1e3:.0f} ms, "
                         f"constructor {t_ctor:.1f} s), OpenMP over particles, gcc -O3"}
        break
    return out


def run_reference(args, pkg) -> dict:
    import torch
    from cpp_fluid_particles_b200 import capi
    solver = args.workload
    libref = os.path.join(ROOT, "oracle", "_ref", "libsphref.so")
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return {}
    scene_name = args.scene or SCENE_OF_N.get(args.gpus, "2m")
    if not (os.path.exists(libref) and torch.cuda.is_available()):
        cb = cpu_baseline(pkg, solver, scene_name if scene_name in ("config0", "200k", "2m") else "2m", budget_s=60.0)
        return {"impl": "reference", "metric": "particle-steps/sec (dam-break)", "value": cb["value"], "unit": cb["unit"],
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
                "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": cb["unit"], "h2d_bytes_per_step": 0,
                                            "d2h_bytes_per_step": 0},
                "config": {"workload": f"{solver} dam-break, CPU restatement (reference CUDA build unavailable here)"}}
    # the reference is single-GPU: at --gpus N its arm runs the SAME scene as this engine's N-GPU arm, on one B200
    sc = pkg.scene.benchmark_scene(scene_name, solver)
    n = sc.fluid.shape[0]
    app = capi.SphApp(sc, libref)
    warm = max(args.warmup, 5)
    steps = args.steps
    for _ in range(warm):
        app.step()
    # Estimator: the MEDIAN of per-step host wall times (SPHSystem::step() synchronises the device before it returns,
    # SPHSystem.cu:142), next to the reference's own cudaEvent figure for the same steps.  The reference allocates and
    # frees device memory inside every Thrust call; those driver calls make single steps jitter by tens of ms (the mean
    # over a short run was not reproducible), and a concurrent nvidia-smi poll contends for the same driver lock -- so
    # nothing polls during the timed loop; clocks are sampled over a second, un-timed run of the same steps.
    torch.cuda.synchronize()
    wall, ms_self = [], []
    t_all = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        ms_self.append(app.step())
        wall.append(time.perf_counter() - t0)
    torch.cuda.synchronize()
    t_all = time.perf_counter() - t_all
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, app.download())
    sampler = ClockSampler(0, period_ms=500); sampler.start()
    for _ in range(steps):
        app.step()
    clocks = sampler.stop()
    app.close()
    dt = float(np.median(wall))
    cb = cpu_baseline(pkg, solver, scene_name if scene_name in ("config0", "200k", "2m") else "2m")
    value = n / dt
    return {"impl": "reference", "metric": "particle-steps/sec (dam-break)", "value": value, "unit": "particle-steps/s",
            "n_gpus": 1, "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3,
            "ms_per_step_estimator": "median of per-step host wall times (each step ends with the reference's own device synchronisation)",
            "ms_per_step_mean_wall": t_all / steps * 1e3, "ms_per_step_min_wall": float(np.min(wall)) * 1e3,
            "ms_per_step_self_reported": float(np.median(ms_self)), "value_self_reported": n / (float(np.median(ms_self)) * 1e-3),
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(scene_name, solver), "engine": "unmodified reference .cu files, nvcc "
                       "-arch=sm_100 --expt-extended-lambda -use_fast_math, on the same B200 (the reference has no CPU path)"},
            "cpu_baseline": {**cb, "note": "CPU restatement; the reference arm's own value is the reference CUDA build",
                             "kind_of_value": "reference"},
            "e2e": {"value": value, "unit": "particle-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "clocks": clocks}


def workload_name(scene_name: str, solver: str) -> str:
    desc = {"dfsph": "DFSPH dt=0.004, 4 divergence + 4 density iterations", "wcsph": "WCSPH dt=0.001",
            "pbd": "PBD dt=0.004, 4 Jacobi projection iterations + XSPH"}[solver]
    return f"{scene_name} dam-break, {desc}"


def timed_kernels(solver: str):
    """(label, method name on SphkSystem, algorithmic bytes key) of the sweeps timed individually."""
    if solver == "dfsph":
        return [("density: computeDensityAlpha + colour gradient + first divergence error (fused sweep)", "fused_density_alpha_div_error",
                 "density_alpha+color_grad+div_error"),
                ("dfsph_div_error", "dfsph_div_error", "dfsph_error"), ("dfsph_div_correct", "dfsph_div_correct", "dfsph_correct"),
                ("dfsph_den_error", "dfsph_den_error", "dfsph_error"), ("dfsph_den_correct", "dfsph_den_correct", "dfsph_correct"),
                ("viscosity + surface (fused sweep)", "fused_viscosity_surface", "viscosity+surface")]
    if solver == "pbd":
        return [("density: pbd_density_lambda", "pbd_density_lambda", "pbd_lambda"),
                ("pbd_delta_pos_apply", "pbd_delta_pos_apply", "pbd_delta_pos"),
                ("pbd_xsph + colour gradient (fused sweep)", "fused_pbd_xsph_color_grad", "pbd_xsph+color_grad"), ("surface", "surface", "surface")]
    return [("density: computeDensity + colour gradient (fused sweep)", "fused_density_color_grad", "density+color_grad"),
            ("pressure_force", "pressure_force", "pressure_force"), ("viscosity + surface (fused sweep)", "fused_viscosity_surface", "viscosity+surface")]


def run_ours_single(args, pkg) -> dict:
    import torch
    from cpp_fluid_particles_b200 import capi, engine
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: this engine has no CPU fallback"
    solver = args.workload
    scene_name = args.scene or "2m"
    sc = pkg.scene.benchmark_scene(scene_name, solver)
    n = sc.fluid.shape[0]
    dev = torch.device("cuda:0")
    # ---------------- device-resident value: python mirror = the same C-ABI calls as the C++ classes ----------
    s = engine.SphkSystem(sc, device=dev)
    ktimes = {}
    evs = {}
    hooks = timed_kernels(solver)

    def wrap(label, meth):
        inner = getattr(s, meth)
        evs[label] = []

        def timed(*a, **k):
            if s._timing and len(evs[label]) < 2 * args.steps * 12:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); r = inner(*a, **k); e1.record()
                evs[label].append((e0, e1))
                return r
            return inner(*a, **k)
        setattr(s, meth, timed)

    s._timing = False
    for label, meth, _ in hooks:
        wrap(label, meth)
    build_evs = []
    inner_build = s.build_neighbor_list

    def timed_build():
        if s._timing:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); inner_build(); e1.record(); build_evs.append((e0, e1))
        else:
            inner_build()
    s.build_neighbor_list = timed_build
    search_evs = []
    inner_search = s.search_fluid

    def timed_search():
        if s._timing:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); inner_search(); e1.record(); search_evs.append((e0, e1))
        else:
            inner_search()
    s.search_fluid = timed_search
    for _ in range(args.warmup):
        s.step()
    launches0 = s.launch_count()
    sampler = ClockSampler(0); sampler.start()
    s._timing = True
    torch.cuda.synchronize()
    e_start, e_stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_start.record()
    for _ in range(args.steps):
        s.step()
    e_stop.record()
    torch.cuda.synchronize()
    s._timing = False
    ms_total = e_start.elapsed_time(e_stop)
    clocks = sampler.stop()
    launches = s.launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, s.state())
    ms_step = ms_total / args.steps
    value = n / (ms_step * 1e-3)
    peak, peak_src = peaks()
    kernels = []
    for label, _, key in hooks:
        t = [a.elapsed_time(b) for a, b in evs[label]]
        if not t:
            continue
        ms = float(np.mean(t))
        gbs = n * ALG_BYTES[key] / (ms * 1e-3) / 1e9
        kernels.append({"kernel": label, "launches_timed": len(t), "ms": ms, "alg_bytes_per_particle": ALG_BYTES[key],
                        "achieved_gbs": gbs, "frac": gbs / peak, "share_of_step": ms * len(t) / args.steps / ms_step})
    t = [a.elapsed_time(b) for a, b in search_evs]
    ms = float(np.mean(t))
    gbs = n * ALG_BYTES["neighbor_search"] / (ms * 1e-3) / 1e9
    kernels.append({"kernel": "neighbor_search (hash+sort+gather+ranges)", "launches_timed": len(t), "ms": ms,
                    "alg_bytes_per_particle": ALG_BYTES["neighbor_search"], "achieved_gbs": gbs, "frac": gbs / peak,
                    "share_of_step": ms / ms_step})
    t = [a.elapsed_time(b) for a, b in build_evs]
    if t:
        kernels.append({"kernel": "neighbor_list_build (27-cell walk, once per step)", "launches_timed": len(t), "ms": float(np.mean(t)),
                        "alg_bytes_per_particle": None, "achieved_gbs": None, "frac": None, "share_of_step": float(np.mean(t)) / ms_step})
    dens = kernels[0]
    stats = s.list_stats()
    traffic, traffic_src = ncu_traffic("OpDensityAlpha") if solver == "dfsph" and scene_name == "2m" else (None, None)
    roof = {"bound": "hbm", "kernel": dens["kernel"], "achieved": dens["achieved_gbs"], "peak": peak, "unit": "GB/s",
            "frac": dens["frac"], "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "alg_bytes_per_launch": n * dens["alg_bytes_per_particle"], "ms_per_launch": dens["ms"], "kernels": kernels,
            "note": "neighbour sweeps are bound by the L1 data pipe (scattered 32-byte-sector gathers) and FP32 issue, "
                    "not by HBM (SURVEY 8d; ncu in profiles/): traffic exceeds the algorithmic bytes by the neighbour list "
                    "streamed once per sweep"}
    if stats:
        roof["neighbors_per_particle"] = stats["total"] / n
    s.close()
    del s
    torch.cuda.empty_cache()
    # ---------------- e2e: C++ class layer through the facade, HOST buffers -------------------------------------------
    # Every step takes a particle state from pinned host memory (H2D pos + vel), runs SPHSystem::step() in the C++ class
    # layer, and returns pos + vel + density to pinned host memory (D2H).  sph_app_submit pipelines the batches: the
    # copies of batch k+1 / k-1 run on a copy stream while batch k steps (include/sph_app.h).  The synchronous variant
    # (upload; step; download with blocking cudaMemcpy, the reference's own idiom) is timed too and reported beside it.
    app = capi.SphApp(sc)
    pin = lambda shape: torch.empty(shape, dtype=torch.float32, pin_memory=True).numpy()  # noqa: E731
    hpos, hvel, hden = pin((n, 3)), pin((n, 3)), pin((n,))
    opos, ovel = pin((n, 3)), pin((n, 3))
    for _ in range(max(3, args.warmup)):     # (the class layer captures its step graph in its third plain step: keep that out of the timed region)
        app.step()
    app.download_into(hpos, hvel, hden)      # the synthetic input batch: the dam-break state after the warm-up steps
    for _ in range(3):
        app.submit(hpos, hvel, opos, ovel, hden)
    app.wait()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        app.submit(hpos, hvel, opos, ovel, hden)   # H2D of this batch + step of the previous one + D2H of its result
    app.wait()                                     # last step + last downloads
    torch.cuda.synchronize()
    e2e_dt = (time.perf_counter() - t0) / args.steps
    assert np.isfinite(hden).all() and np.isfinite(opos).all()
    # synchronous variant
    t0 = time.perf_counter()
    for _ in range(args.steps):
        app.upload(hpos, hvel); app.step(); app.download_into(opos, ovel, hden)
    torch.cuda.synchronize()
    sync_dt = (time.perf_counter() - t0) / args.steps
    app.close()
    e2e = {"value": n / e2e_dt, "unit": "particle-steps/s", "ms_per_step": e2e_dt * 1e3, "h2d_bytes_per_step": 24 * n,
           "d2h_bytes_per_step": 28 * n,
           "api": "SPHSystem (C++ class layer) via the sph_app facade: sph_app_submit / sph_app_wait, pinned host buffers, "
                  "copies on a copy stream overlapped with the previous batch's step",
           "timer": "host wall clock over K submits + the final wait (every upload, step and download inside)",
           "synchronous_ms_per_step": sync_dt * 1e3, "synchronous_value": n / sync_dt,
           "synchronous_api": "sph_app_upload_fluid; sph_app_step; sph_app_download_fluid with blocking cudaMemcpy"}
    cb = cpu_baseline(pkg, solver, scene_name if scene_name in ("config0", "200k", "2m") else "2m")
    return {"metric": "particle-steps/sec (dam-break)", "value": value, "unit": "particle-steps/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(scene_name, solver), "n_fluid": n, "n_boundary": int(sc.boundary.shape[0]),
                       "cells": list(sc.params.cell_size), "l2": "inputs larger than L2: packed particles + neighbour list "
                       "working set per sweep is ~%d MB > 126 MB L2; no flush between steps" % int(n * (32 + 36 * 4) / 1e6),
                       "parallelism": "1 GPU",
                       "value_api": "python mirror of the C++ class layer (engine.SphkSystem: the same C-ABI calls in the same order, "
                                    "bit-identical by test_python_mirror_equals_class_layer); e2e runs through the C++ classes"},
            "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cb, "clocks": clocks}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="dfsph", choices=["dfsph", "wcsph", "pbd"])
    ap.add_argument("--scene", default=None, help="override the scene (mini, config0, 200k, 2m, ...)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (default, the driver's contract): 2M fluid particles per GPU, N=8 is BASELINE configs[4]; "
                         "strong: the same scene (--scene, default 2m) split over N GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the state after the last timed step as DIR/<name>.npy (single-GPU runs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    args.warmup = max(args.warmup, 3)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (world > 1 or args.gpus > 1) and args.impl == "ours":
        ap.error("--dump-outputs writes the single-GPU path's outputs: use it with --gpus 1")
    import pkgload
    pkg = pkgload.load()
    if args.impl == "reference":
        out = run_reference(args, pkg)
        if out:
            print(json.dumps(out), flush=True)
        return
    if world > 1 or args.gpus > 1:
        from cpp_fluid_particles_b200 import slabs
        out = slabs.bench_main(args, pkg)
        if out:
            print(json.dumps(out), flush=True)
        return
    print(json.dumps(run_ours_single(args, pkg)), flush=True)


if __name__ == "__main__":
    main()
