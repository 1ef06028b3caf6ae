"""Generates the golden fixtures from the REFERENCE's own CUDA kernels (oracle/_ref/libsphref.so: the
unmodified reference .cu files compiled for sm_100 with the reference's flags by oracle/ref_build/Makefile).
The reference has no CPU path, so this runs on a GPU, from a tree where __graft_entry__.build() found the
reference sources:

    python tests/golden/make_golden.py OUT_DIR

and the produced files are then copied into tests/golden/ and committed.

  mini_<solver>.npz   scene "mini" (1 400 fluid + 3 752 boundary particles, same generator and constants as
                      config 0), fixed-work solver settings of BASELINE.md: full state after the constructor
                      (step 0, Q3) and after each of 2 explicit steps
  meta.json           rcp.approx(cellLength) of the device, which lets the CPU oracle reproduce the GPU hash
  reference_cuda.npz  what tests/test_gpu_system.py compares the class layer against, for scenes too large to
                      store whole: per state the sha256 of every array compared bit for bit (keys, sorted
                      positions), and ROWS fixed, seeded rows of every field compared with a tolerance together
                      with max |field| over all particles (the scale of util.relerr)
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pkgload  # noqa: E402
from util import cell_start_from_p2c, digest  # noqa: E402

pkg = pkgload.load()
from cpp_fluid_particles_b200 import capi, engine  # noqa: E402

out = sys.argv[1]
os.makedirs(out, exist_ok=True)
LIBREF = os.path.join(ROOT, "oracle", "_ref", "libsphref.so")
STEPS = 2
ROWS = 128
SOLVERS = ("wcsph", "dfsph", "pbd")
meta = {}
for solver in SOLVERS:
    sc = pkg.scene.benchmark_scene("mini", solver)
    app = capi.SphApp(sc, LIBREF)
    assert app.engine == "reference-cuda"
    data = {"steps": np.int32(STEPS)}
    for k in range(STEPS + 1):
        st = app.download()
        data[f"pos_{k}"], data[f"density_{k}"], data[f"p2c_{k}"] = st["pos"], st["density"], st["p2c"]
        data[f"vel_{k}"] = st["vel"]
        if k < STEPS:
            app.step()
    b = app.download_boundary()
    data["massB"], data["p2cB"] = b["mass"], b["p2c"]
    np.savez_compressed(os.path.join(out, f"mini_{solver}.npz"), **data)
    app.close()
probe = engine.SphkSystem(pkg.scene.make_scene("mini"), step0=False)
rcp = probe.device_rcp(pkg.scene.make_scene("mini").params.cell_length)
meta["rcp_cell_length_bits"] = int(np.float32(rcp).view(np.uint32))
meta["cell_length"] = float(pkg.scene.make_scene("mini").params.cell_length)
import torch  # noqa: E402
meta["device"] = torch.cuda.get_device_name(0)
with open(os.path.join(out, "meta.json"), "w") as f:
    json.dump(meta, f, indent=1)

# ---- reference_cuda.npz ----------------------------------------------------------------------------------------------
gold = {}


def rows(case, n, seed):
    idx = np.sort(np.random.default_rng(seed).choice(n, size=min(n, ROWS), replace=False)).astype(np.int64)
    gold[case + ".idx"] = idx
    return idx


def record(key, st, idx, fields=(), digests=()):
    for f in fields:
        gold[f"{key}.{f}"] = st[f][idx]
        gold[f"{key}.{f}.scale"] = np.float64(np.abs(st[f].astype(np.float64)).max())
    for f in digests:
        gold[f"{key}.{f}.sha256"] = np.str_(digest(st[f]))


def record_boundary(case, app, seed):
    b = app.download_boundary()
    record(case + "-boundary", b, rows(case + "-boundary", b["mass"].shape[0], seed), ("mass",), ("p2c", "pos"))


seed = 0
FIELDS = ("pos", "density", "vel", "pressure")
# test_class_layer_vs_reference_cuda: config0, plain and jittered lattice, constructor + 3 steps
for solver in SOLVERS:
    for name, jitter in (("config0", 0.0), ("config0", 0.001)):
        sc = pkg.scene.benchmark_scene(name, solver)
        if jitter:
            sc = pkg.scene.make_scene(name, solver=solver, dt=sc.params.dt, max_iter=sc.params.max_iter,
                                      den_thr=sc.params.density_error_threshold, div_thr=sc.params.divergence_error_threshold,
                                      jitter=jitter)
        case = f"{name}{'-jitter' if jitter else ''}-{solver}"
        app = capi.SphApp(sc, LIBREF)
        seed += 1
        idx = rows(case, app.nF, seed)
        for k in range(4):
            record(f"{case}.s{k}", app.download(), idx, FIELDS, ("p2c", "pos"))
            app.step()
        seed += 1
        record_boundary(case, app, seed)
        app.close()
# test_class_layer_vs_reference_cuda_200k: constructor + 2 steps
app = capi.SphApp(pkg.scene.benchmark_scene("200k", "dfsph"), LIBREF)
seed += 1
idx = rows("200k-dfsph", app.nF, seed)
for k in range(3):
    record(f"200k-dfsph.s{k}", app.download(), idx, FIELDS, ("p2c",))
    app.step()
app.close()
# test_class_layer_vs_reference_cuda_2m: boundary, constructor + 1 step
for solver in SOLVERS:
    sc = pkg.scene.benchmark_scene("2m", solver)
    case = f"2m-{solver}"
    app = capi.SphApp(sc, LIBREF)
    seed += 1
    record_boundary(case, app, seed)
    seed += 1
    idx = rows(case, app.nF, seed)
    for k in range(2):
        st = app.download()
        st["cell_start"] = cell_start_from_p2c(st["p2c"], sc.params.ncells)
        record(f"{case}.s{k}", st, idx, ("pos", "density"), ("p2c", "cell_start", "pos"))
        app.step()
    app.close()
# test_sorted_order_bit_exact_through_steps: mini, 6 steps
for solver in SOLVERS:
    sc = pkg.scene.benchmark_scene("mini", solver)
    app = capi.SphApp(sc, LIBREF)
    for k in range(6):
        app.step()
        st = app.download()
        st["cell_start"] = cell_start_from_p2c(st["p2c"], sc.params.ncells)
        record(f"mini-{solver}.s{k}", st, None, (), ("p2c", "cell_start"))
    app.close()
gold["device"] = np.str_(meta["device"])
np.savez_compressed(os.path.join(out, "reference_cuda.npz"), **gold)
print("golden written to", out, meta, f"{len(gold)} arrays in reference_cuda.npz")
