"""Whole-step parity on the GPU:
  * the C++ class layer (libsphhost.so, through the reference's own call sites restated in sph_app.cpp)
    against the reference's own CUDA kernels (the unmodified reference .cu files compiled for sm_100, run on a
    B200 by tests/golden/make_golden.py, outputs stored in tests/golden/reference_cuda.npz) on identical inputs:
    bit-exact particle2cell / sort order / cellStart (sha256 over all particles), <= 1e-5 scale-relative on
    positions and densities after the constructor (step 0, Q3) and after each explicit step (on stored rows);
  * the same against the CPU restatement (oracle/) and against the committed golden fixtures;
  * the python mirror (engine.SphkSystem) against the C++ layer (must be identical: same C-ABI calls).
"""
import os

import numpy as np
import pytest

from util import GOLDEN, TOL, assert_close, assert_close_sample, bits, cell_start_from_p2c, digest, relerr

pytestmark = pytest.mark.gpu

SOLVERS = ["wcsph", "dfsph", "pbd"]


def _gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("pytest -m gpu needs a CUDA device: libsphk has no CPU fallback")


@pytest.fixture(scope="module")
def gold():
    """Outputs of the reference's own CUDA kernels (tests/golden/make_golden.py)."""
    with np.load(os.path.join(GOLDEN, "reference_cuda.npz")) as z:
        return {k: z[k] for k in z.files}


def _same_bits(a, gold, key):
    return digest(a) == str(gold[key + ".sha256"])


def _run(app, steps):
    out = [app.download()]
    for _ in range(steps):
        app.step()
        out.append(app.download())
    return out


def _compare_states(ours, gold, key, what, vel_tol=2e-4):
    assert _same_bits(ours["p2c"], gold, key + ".p2c"), f"{what}: particle2cell differs"
    assert_close_sample(ours["pos"], gold, key + ".pos", what=f"{what} pos")
    assert_close_sample(ours["density"], gold, key + ".density", what=f"{what} density")
    assert_close_sample(ours["vel"], gold, key + ".vel", tol=vel_tol, what=f"{what} vel")
    assert_close_sample(ours["pressure"], gold, key + ".pressure", tol=1e-4, what=f"{what} pressure")


def _compare_boundary(app, gold, case):
    b, key = app.download_boundary(), case + "-boundary"
    assert _same_bits(b["p2c"], gold, key + ".p2c")
    assert _same_bits(b["pos"], gold, key + ".pos"), "sorted boundary positions must be bit-identical"
    assert_close_sample(b["mass"], gold, key + ".mass", what=f"{case} boundary mass")


@pytest.mark.parametrize("solver", SOLVERS)
@pytest.mark.parametrize("name,jitter", [("config0", 0.0), ("config0", 0.001)])
def test_class_layer_vs_reference_cuda(pkg, built, gold, solver, name, jitter):
    _gpu()
    from cpp_fluid_particles_b200 import capi
    sc = pkg.scene.benchmark_scene(name, solver)
    if jitter:
        sc = pkg.scene.make_scene(name, solver=solver, dt=sc.params.dt, max_iter=sc.params.max_iter,
                                  den_thr=sc.params.density_error_threshold, div_thr=sc.params.divergence_error_threshold,
                                  jitter=jitter)
    case = f"{name}{'-jitter' if jitter else ''}-{solver}"
    ours_app = capi.SphApp(sc)
    assert ours_app.engine == "b200-native"
    ours = _run(ours_app, 3)
    # boundary set: searched once in the constructor
    _compare_boundary(ours_app, gold, case)
    for k, o in enumerate(ours):
        if solver == "pbd" and k == 0:
            # Q6: PBD's step 0 is neighbour search + posLast init only -> pure sort: bit-identical order
            assert _same_bits(o["pos"], gold, f"{case}.s0.pos"), "sort permutation differs from the reference"
        _compare_states(o, gold, f"{case}.s{k}", f"{solver} after step {k}")
    ours_app.close()


def test_class_layer_vs_reference_cuda_200k(pkg, built, gold):
    """A denser check at 216 000 fluid + 58 808 boundary particles (DFSPH 4+4): two steps against the reference's
    own kernels."""
    _gpu()
    from cpp_fluid_particles_b200 import capi
    sc = pkg.scene.benchmark_scene("200k", "dfsph")
    a = capi.SphApp(sc)
    for k in range(3):
        _compare_states(a.download(), gold, f"200k-dfsph.s{k}", f"200k dfsph step {k}")
        a.step()
    a.close()


@pytest.mark.parametrize("solver", SOLVERS)
def test_class_layer_vs_reference_cuda_2m(pkg, built, gold, solver):
    """BASELINE.json configs[1-3] at their real size (2 097 152 fluid + 237 608 boundary particles): the C++ class
    layer against the reference's own CUDA kernels -- constructor state (step 0, Q3) and one explicit step.
    Bit-exact particle2cell / cellStart / sorted boundary; <= 1e-5 scale-relative on positions and densities, and
    <= 1e-5 PER ELEMENT on the densities of interior particles (rho >= 0.9 rho0: no free-surface cancellation) among
    the stored rows."""
    _gpu()
    from cpp_fluid_particles_b200 import capi
    sc = pkg.scene.benchmark_scene("2m", solver)
    case = f"2m-{solver}"
    a = capi.SphApp(sc)
    _compare_boundary(a, gold, case)
    nc = sc.params.ncells
    idx = gold[case + ".idx"]
    for k in range(2):
        sa, key = a.download(), f"{case}.s{k}"
        assert _same_bits(sa["p2c"], gold, key + ".p2c"), f"2m {solver} step {k}: particle2cell differs"
        assert _same_bits(cell_start_from_p2c(sa["p2c"], nc), gold, key + ".cell_start")
        assert_close_sample(sa["pos"], gold, key + ".pos", what=f"2m {solver} step {k} pos")
        assert_close_sample(sa["density"], gold, key + ".density", what=f"2m {solver} step {k} density")
        if solver == "pbd" and k == 0:
            assert _same_bits(sa["pos"], gold, key + ".pos"), "sort permutation differs from the reference"
        ref_d = gold[key + ".density"]
        interior = ref_d >= 0.9 * sc.params.rho0
        if interior.any():
            d = np.abs(sa["density"][idx][interior].astype(np.float64) - ref_d[interior]) / ref_d[interior]
            assert d.max() <= 1e-5, f"2m {solver} step {k}: per-element interior density error {d.max():.2e}"
        a.step()
    a.close()


@pytest.mark.parametrize("solver", SOLVERS)
def test_sorted_order_bit_exact_through_steps(pkg, built, gold, solver):
    """The stable-sort permutation and cellStart stay identical to the reference while the fluid moves:
    particle2cell of step k is computed from positions that already differ by ~1e-7, so exact equality of
    the keys over several steps is a strong check of both the physics and the hash."""
    _gpu()
    from cpp_fluid_particles_b200 import capi
    sc = pkg.scene.benchmark_scene("mini", solver)
    a = capi.SphApp(sc)
    for k in range(6):
        a.step()
        sa = a.download()
        assert _same_bits(sa["p2c"], gold, f"mini-{solver}.s{k}.p2c"), f"step {k}"
        nc = sc.params.ncells
        assert _same_bits(cell_start_from_p2c(sa["p2c"], nc), gold, f"mini-{solver}.s{k}.cell_start")
    a.close()


@pytest.mark.parametrize("solver", SOLVERS)
def test_class_layer_vs_cpu_oracle(pkg, built, solver):
    _gpu()
    from cpp_fluid_particles_b200 import capi, engine
    from oracle import oracle as O
    sc = pkg.scene.benchmark_scene("config0", solver)
    app = capi.SphApp(sc)
    probe = engine.SphkSystem(pkg.scene.make_scene("mini"), step0=False)
    rcp = probe.device_rcp(sc.params.cell_length)
    probe.close()
    osys = O.OracleSystem(sc, hash_rcp=rcp)
    for k in range(3):
        st = app.download()
        assert np.array_equal(st["p2c"], osys.field("p2c")), f"step {k} p2c"
        assert_close(st["pos"], osys.field("pos"), what=f"{solver} step {k} pos")
        assert_close(st["density"], osys.field("density"), what=f"{solver} step {k} density")
        assert_close(st["vel"], osys.field("vel"), tol=5e-4, what=f"{solver} step {k} vel")
        app.step(); osys.step()
    app.close(); osys.close()


@pytest.mark.parametrize("solver", SOLVERS)
@pytest.mark.parametrize("use_list", [True, False])
def test_python_mirror_equals_class_layer(pkg, built, solver, use_list):
    """engine.SphkSystem and the C++ classes issue the same C-ABI calls -> identical bits (list path on);
    with the list off (pure cell walk) results may differ only by the contribution-free candidates."""
    _gpu()
    from cpp_fluid_particles_b200 import capi, engine
    sc = pkg.scene.benchmark_scene("mini", solver)
    app = capi.SphApp(sc)
    s = engine.SphkSystem(sc, use_list=use_list)
    for k in range(3):
        a, b = app.download(), s.state()
        assert np.array_equal(a["p2c"], b["p2c"])
        if use_list:
            assert np.array_equal(bits(a["pos"]), bits(b["pos"])), f"{solver} step {k}"
            assert np.array_equal(bits(a["density"]), bits(b["density"]))
        else:       # same pairs, same order, but another kernel instantiation (FMA contraction may differ)
            assert_close(b["pos"], a["pos"], tol=1e-6, what=f"{solver} step {k} pos")
            assert_close(b["density"], a["density"], tol=1e-6, what=f"{solver} step {k} density")
        app.step(); s.step()
    app.close(); s.close()


@pytest.mark.parametrize("solver", SOLVERS)
def test_against_golden_fixtures(pkg, built, solver):
    """Committed outputs of the reference's own CUDA kernels (tests/golden/make_golden.py, run on a B200)."""
    _gpu()
    path = os.path.join(GOLDEN, f"mini_{solver}.npz")
    if not os.path.exists(path):
        pytest.skip("golden fixture not generated yet")
    from cpp_fluid_particles_b200 import capi
    gold = np.load(path)
    sc = pkg.scene.benchmark_scene("mini", solver)
    app = capi.SphApp(sc)
    for k in range(int(gold["steps"]) + 1):
        st = app.download()
        assert np.array_equal(st["p2c"], gold[f"p2c_{k}"]), f"step {k} p2c"
        assert_close(st["pos"], gold[f"pos_{k}"], what=f"golden {solver} step {k} pos")
        assert_close(st["density"], gold[f"density_{k}"], what=f"golden {solver} step {k} density")
        app.step()
    app.close()


@pytest.mark.parametrize("solver", ["wcsph", "dfsph", "pbd"])
def test_fused_sweeps_equal_per_launch_site_path(pkg, built, solver):
    """The fused sweeps (default) against one kernel per reference launch site: same quantities, same order of
    operations per quantity -> equal up to FMA contraction between kernel instantiations."""
    _gpu()
    from cpp_fluid_particles_b200 import engine
    sc = pkg.scene.benchmark_scene("config0", solver)
    a, b = engine.SphkSystem(sc, step0=False), engine.SphkSystem(sc, step0=False)
    b.fused = False
    for k in range(4):
        a.step(); b.step()
        sa, sb = a.state(), b.state()
        assert np.array_equal(sa["p2c"], sb["p2c"])
        assert_close(sa["pos"], sb["pos"], tol=1e-6, what=f"{solver} step {k} pos")
        assert_close(sa["density"], sb["density"], tol=1e-6, what=f"{solver} step {k} density")
        assert_close(sa["vel"], sb["vel"], tol=1e-5, what=f"{solver} step {k} vel")
    assert a.launch_count() < b.launch_count()
    a.close(); b.close()


@pytest.mark.parametrize("name,jitter", [("mini", 0.0), ("config0", 0.002)])
def test_dfsph_adaptive_device_loops(pkg, built, name, jitter):
    """Default DFSPH (thresholds 1e-3, max 20 iterations; DFSPHSolver.h:27-30, the reference's own main.cpp:125 path).
    The loop tests of DFSPHSolver.cu:187,347 run on the device (sphk_loop_*): no error sum is read back, the step is a
    fixed launch sequence and is replayed as a CUDA graph.  Checked against
      (a) the same engine with the reference's host loop (one reduction read back per iteration): identical iteration
          counts and identical bits -- the device evaluates the same test on the same sums;
      (b) the CPU oracle: iteration counts within +-1 (the reduction order differs) and state <= 1e-5."""
    _gpu()
    from cpp_fluid_particles_b200 import capi, engine
    from oracle import oracle as O
    sc = pkg.scene.make_scene(name, solver="dfsph", dt=0.004, jitter=jitter)
    dev, host = capi.SphApp(sc), capi.SphApp(sc)
    host.set_option(1, 0)
    probe = engine.SphkSystem(pkg.scene.make_scene("mini"), step0=False)
    rcp = probe.device_rcp(sc.params.cell_length)
    probe.close()
    osys = O.OracleSystem(sc, hash_rcp=rcp)
    for k in range(6):
        ms = dev.step(); host.step(); osys.step()
        assert ms > 0
        a, b = dev.download(), host.download()
        it_dev, it_host = dev.dfsph_iterations(), host.dfsph_iterations()
        assert it_dev == it_host, f"step {k}: device loop ran {it_dev} iterations, host loop {it_host}"
        assert 1 <= it_dev[0] <= 20 and 2 <= it_dev[1] <= 20
        assert np.array_equal(bits(a["pos"]), bits(b["pos"])) and np.array_equal(bits(a["density"]), bits(b["density"]))
        it_o = (O.lib().oracle_system_iters(osys.h, 0), O.lib().oracle_system_iters(osys.h, 1))
        assert abs(it_dev[0] - it_o[0]) <= 1 and abs(it_dev[1] - it_o[1]) <= 1, f"step {k}: {it_dev} vs oracle {it_o}"
        if it_dev == it_o:
            assert_close(a["pos"], osys.field("pos"), what=f"adaptive dfsph step {k} pos")
            assert_close(a["density"], osys.field("density"), what=f"adaptive dfsph step {k} density")
    dev.close(); host.close(); osys.close()


def test_full_size_properties_2m(pkg, built):
    """BASELINE.json's full size (2M fluid particles): size-independent properties instead of the oracle:
    cellStart is the exclusive scan of the key histogram, sorted order is non-decreasing in key, the
    permutation is a bijection, densities of interior lattice particles equal the analytic lattice sum."""
    _gpu()
    import torch
    from cpp_fluid_particles_b200 import engine
    sc = pkg.scene.benchmark_scene("2m", "dfsph")
    s = engine.SphkSystem(sc, step0=False)
    n, nc = s.fluid.n, sc.params.ncells
    p2c = s.fluid.p2c.cpu().numpy()
    cs = s.cs_fluid.cpu().numpy()
    assert np.array_equal(cs, cell_start_from_p2c(p2c, nc))
    perm = s.permutation().cpu().numpy()
    assert np.array_equal(np.sort(perm), np.arange(n, dtype=np.int32))
    keys_sorted = p2c[perm]
    assert np.all(np.diff(keys_sorted) >= 0), "sortedness"
    same = np.diff(keys_sorted) == 0
    assert np.all(np.diff(perm)[same] > 0), "stability: equal keys keep their previous relative order"
    assert np.array_equal(bits(s.fluid.pos.cpu().numpy()), bits(sc.fluid[perm]))
    s.dfsph_density_alpha()
    dens = s.fluid.density.cpu().numpy()
    # interior particle of the 0.02 lattice with R = 0.04: analytic lattice sum (self excluded, Q1)
    from oracle import oracle as O
    mini = pkg.scene.make_scene("config0")
    g = O.grid(mini.params.cell_size, mini.params.cell_length)
    ps, _, _, csm, _ = O.neighbor_search(mini.fluid, np.zeros_like(mini.fluid), g)
    pb, _, _, csb, _ = O.neighbor_search(mini.boundary, None, g)
    A = O.SceneArrays(ps, np.full(ps.shape[0], mini.params.m0, np.float32), csm, pb, np.zeros(pb.shape[0], np.float32), csb, g, mini.params.radius)
    ref_d = O.density(A)
    interior = float(np.median(ref_d[ref_d > 0.99 * ref_d.max()]))
    assert abs(float(np.median(dens[dens > 0.99 * dens.max()])) - interior) <= 1e-5 * interior
    stats = s.list_stats()
    assert stats["overflow"] == 0
    # idempotence: searching again on sorted input is the identity permutation
    s.search_fluid()
    assert np.array_equal(s.permutation().cpu().numpy(), np.arange(n, dtype=np.int32))
    s.step(); s.step()
    st_pos = s.fluid.pos.cpu().numpy()
    assert np.isfinite(st_pos).all() and st_pos.min() >= 0 and st_pos.max() <= 0.99 * sc.params.space[0] + 1e-6
    s.close()


@pytest.mark.parametrize("solver,iters", [("dfsph", 4), ("sph", 0), ("pbd", 4)])
def test_headless_cli_matches_facade(pkg, built, tmp_path, solver, iters):
    """SURVEY 8f-1: the reference application without its window (app/sph_headless.cpp, C++ against the class API only)
    run as a process -- constructor + 3 frames, particle dump -- against capi.SphApp on the same scene: the same engine
    behind two independent restatements of main.cpp's call sites, so the dumps must agree bit for bit; also checks the
    timing line / JSON summary of oneStep() (main.cpp:300-306)."""
    _gpu()
    import json
    import subprocess
    from util import ROOT
    from cpp_fluid_particles_b200 import capi
    cli = os.path.join(ROOT, "cpp-fluid-particles_b200", "sph_headless")
    assert os.path.exists(cli), "sph_headless is not built"
    pyname = {"sph": "wcsph"}.get(solver, solver)
    sc = pkg.scene.benchmark_scene("mini", pyname)
    box, (nx, ny, nz), origin = pkg.scene._CONFIGS["mini"]
    prefix = str(tmp_path / "dump")
    cmd = [cli, "--solver", solver, "--frames", "3", "--box", str(box), "--block", str(nx), str(ny), str(nz),
           "--origin", *[repr(float(o)) for o in origin], "--dump", prefix, "--quiet"]
    if iters:
        cmd += ["--iters", str(iters)]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    summary = json.loads(out.stdout.strip().splitlines()[-1])
    assert summary["n_fluid"] == sc.fluid.shape[0] and summary["n_boundary"] == sc.boundary.shape[0]
    assert summary["frames"] == 3 and summary["avg_ms_per_frame"] > 0 and summary["particle_steps_per_s"] > 0
    app = capi.SphApp(sc)
    for _ in range(3):
        app.step()
    st = app.download()
    app.close()
    pos = np.fromfile(prefix + ".pos.f32", np.float32).reshape(-1, 3)
    den = np.fromfile(prefix + ".density.f32", np.float32)
    rgb = np.fromfile(prefix + ".rgb.f32", np.float32).reshape(-1, 3)
    assert np.array_equal(bits(pos), bits(st["pos"])), "CLI and facade drive the same engine through the same call sites"
    assert np.array_equal(bits(den), bits(st["density"]))
    assert rgb.shape == pos.shape and np.isfinite(rgb).all() and rgb.min() >= 0.0 and rgb.max() <= 1.0


@pytest.mark.parametrize("solver", ["dfsph", "wcsph"])
def test_pipelined_host_buffer_stepping(pkg, built, solver):
    """sph_app_submit / sph_app_wait (uploads and downloads overlapped with the previous batch's step) against the blocking
    upload; step; download sequence on the same batches: identical bits, batch by batch."""
    _gpu()
    import torch
    from cpp_fluid_particles_b200 import capi
    sc = pkg.scene.benchmark_scene("config0", solver)
    n = sc.fluid.shape[0]
    a, b = capi.SphApp(sc), capi.SphApp(sc)
    for _ in range(3):
        a.step(); b.step()
    pin = lambda shape: torch.empty(shape, dtype=torch.float32, pin_memory=True).numpy()  # noqa: E731
    hpos, hvel = pin((n, 3)), pin((n, 3))
    a.download_into(hpos, hvel, None)
    want, got = [], [(pin((n, 3)), pin((n, 3)), pin((n,))) for _ in range(5)]
    for k in range(5):
        a.upload(hpos, hvel); a.step()
        st = a.download()
        want.append((st["pos"].copy(), st["vel"].copy(), st["density"].copy()))
    for k in range(5):
        b.submit(hpos, hvel, *got[k])
    b.wait()
    for k in range(5):
        for w, g, f in zip(want[k], got[k], ("pos", "vel", "density")):
            assert np.array_equal(bits(w), bits(g)), f"batch {k} {f}"
    a.close(); b.close()
