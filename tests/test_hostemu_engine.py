"""The engine's own sources -- mvicp.cu and every kernel header -- compiled by g++ against the miniature CUDA model in
tools/hostemu (TEST INFRASTRUCTURE: fibers for CTA threads, host memory for device memory) and driven through the same C ABI
and the same parity tests as the GPU suite, at small sizes.  This exercises the LOGIC of the whole device path (search,
median select, residual/Jacobian reduction, LM state machine, general path, normals) on the CPU; the hardware's roundings,
memory model and the multi-GPU exchange are covered only by `pytest -m gpu`.  The product never loads this library."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools", "hostemu"))


@pytest.fixture(scope="module", params=["ascending", "random"])
def emu(request, tmp_path_factory):
    """Builds libmvicp_hostemu.so and points the ctypes binding at it for the duration of this module.  Second pass: the
    threads of a CTA run in a fresh pseudo-random order between any two barriers (HOSTEMU_ORDER=random), so code that lacks a
    barrier cannot pass both; the slow cases run in the first pass only."""
    import shutil
    import build_hostemu
    from mv_lm_icp_b200 import _lib
    so = build_hostemu.build()
    if request.param == "random":       # the order is read once when the library is loaded: load a private copy
        so2 = str(tmp_path_factory.mktemp("hostemu") / "libmvicp_hostemu_random.so")
        shutil.copy(so, so2); so = so2
        os.environ["HOSTEMU_ORDER"] = "random"
    lib = C.CDLL(so); lib.mvicp_last_error.restype = C.c_char_p
    os.environ.pop("HOSTEMU_ORDER", None)
    lib.order = request.param
    saved = _lib._lib
    _lib._lib = lib
    yield lib
    _lib._lib = saved


def _first_pass_only(emu):
    if emu.order != "ascending":
        pytest.skip("slow case: first pass only")


def test_exports_every_abi_symbol(emu):
    from mv_lm_icp_b200 import _lib
    for name in _lib.EXPORTS:
        assert hasattr(emu, name), name


def test_correspondence_step(emu, oracle, golden_dir):
    import test_gpu_corr as T
    T.test_synthetic_bit_exact(oracle, 4, 5000, 21)
    T.test_seed_and_schedule_do_not_change_results(oracle)
    T.test_real_bunny_pair_fp64_storage(oracle, golden_dir)
    import test_gpu_zz_dinosaur as TD
    TD.test_real_dinosaur_pair_mm_units(golden_dir)
    T.test_edge_cases(oracle)
    T.test_median_with_masses_of_near_equal_distances(oracle)
    T.test_closest_point_api(oracle)
    T.test_all_edges_in_one_call_equal_the_per_edge_lists(oracle)
    T.test_guessed_median_select_is_exact(oracle)
    T.test_cutoff_boundary_is_the_reference_comparison(oracle)
    T.test_guessed_median_select_degenerate_buckets(oracle)
    T.test_certified_matches_are_exact(oracle)
    T.test_certificates_with_ties_and_duplicates(oracle)


@pytest.mark.parametrize("param", [0, 1, 2])
@pytest.mark.parametrize("cost", [0, 1, 2])
@pytest.mark.parametrize("robust", [False, True])
def test_lm_step_matches_oracle(emu, oracle, golden_dir, param, cost, robust):
    import test_gpu_lm as T
    if emu.order != "ascending" and (param, cost, robust) not in ((2, 1, True), (1, 0, False), (0, 2, True)):
        pytest.skip("second pass: three configurations")
    T.test_optimize_matches_oracle(oracle, golden_dir, param, cost, robust)


def test_lm_pipeline_pairwise_and_general_path(emu, oracle, golden_dir):
    import test_gpu_lm as T
    if emu.order != "ascending":        # second pass: the general (non-unit quaternion) path only
        T.test_real_bunny_nonrigid_poses(oracle, golden_dir, 2, 1)
        return
    T.test_pipeline_round_matches_oracle(oracle)
    T.test_frame0_is_fixed_inside_the_optimiser()
    T.test_quaternion_parameterisation_drifts_off_the_unit_sphere(oracle)
    for name, param, cost in (("pointToPoint_CeresAngleAxis", 0, 0), ("pointToPoint_EigenQuaternion", 1, 0), ("pointToPoint_SophusSE3", 2, 0),
                              ("pointToPlane_CeresAngleAxis", 0, 1), ("pointToPlane_EigenQuaternion", 1, 1), ("pointToPlane_SophusSE3", 2, 1)):
        T.test_pairwise_known_answer(oracle, golden_dir, name, param, cost)
    T.test_real_bunny_nonrigid_poses(oracle, golden_dir, 2, 1)      # non-unit quaternions: general frame model
    T.test_real_bunny_nonrigid_poses(oracle, golden_dir, 1, 0)


@pytest.mark.parametrize("n_views", [29, 40])
def test_lm_many_views_global_factor(emu, oracle, n_views):
    import test_gpu_lm as T
    if n_views == 40:
        _first_pass_only(emu)
    T.test_many_views_factor_in_global_memory(oracle, n_views)


def test_solver_edges(emu, oracle, golden_dir):
    """tests/test_gpu_solver_edges.py at small sizes: fixed frames anywhere, the factor crossing the shared-memory limit, every
    option set and termination, a weight-0 robust edge, knn_self / normals at every k, fixed flags toggled in certified rounds."""
    import test_gpu_solver_edges as T
    first = emu.order == "ascending"
    for mask in T.MASKS:
        for param, cost in (((0, 0), (1, 2), (2, 1)) if first else ((2, 2),)):
            T.check_fixed_frames(oracle, mask, param, cost, n_points=1000)
    for name, *_ in T.OPTION_SETS:
        for param in ((0, 2) if first else (2,)):
            T.check_option_set(oracle, name, param, n_points=1500)
    T.check_options_general_path(oracle, golden_dir)
    T.check_weight0_pipeline(oracle, n_points=1500)
    for f32 in (True, False):
        T.check_knn_self(f32, big=3001 if first else 0, sample=100)
    T.check_normals_every_k(oracle, n_points=2000)
    T.check_fixed_toggle_in_converged_rounds(oracle, n_views=5, n_points=2003, warm=6)
    if first:
        T.check_factor_crosses_shared_memory(oracle, n_points=300)


def test_normals(emu, oracle, golden_dir):
    import test_gpu_normals as T
    T.test_normals_match_oracle_synthetic(oracle)
    if emu.order == "ascending":
        T.test_normals_real_scan_and_lm_uses_them(oracle, golden_dir)


def test_headless_driver_on_the_emulated_engine(emu, tmp_path):
    """apps/multiview_main.cpp linked against the emulated library: the reference's file formats, flags and loop end to end,
    bit-identical to the Python mirror of the same loop (what tests/test_app_multiview.py checks on the GPU)."""
    import subprocess
    import test_app_multiview as A
    _first_pass_only(emu)
    from helpers import scene
    from mv_lm_icp_b200 import Frame, ICP_Ceres
    build_dir = os.path.join(ROOT, "tools", "hostemu", "_build")
    exe = os.path.join(build_dir, "multiview_hostemu")
    subprocess.run(["/usr/bin/g++", "-O2", "-std=c++11", "-o", exe, os.path.join(ROOT, "apps", "multiview_main.cpp"), "-L" + build_dir,
                    "-lmvicp_hostemu", "-Wl,-rpath," + build_dir], check=True)
    sc = scene(4, 1500, 17)
    A._write_scene(str(tmp_path), sc)
    out = tmp_path / "out"; out.mkdir()
    r = subprocess.run([exe, f"--dir={tmp_path}", "--step=1", "--knn=2", "--rounds=3", f"--out={out}"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    got = [np.loadtxt(out / f"pose_out_{i}.txt") for i in range(4)]
    frames = [Frame(p, n, pose=P) for p, n, P in zip(sc["pts"], sc["nor"], sc["poses_init"])]
    icp = ICP_Ceres(frames)
    icp.recomputeNormals(10)
    frames[0].fixed = True
    icp.computePoseNeighbours(2)
    for _ in range(3):
        icp.computeClosestPoints(0.05)
        icp.ceresOptimizer_sophusSE3(True, True)
    for i in range(4):
        assert np.array_equal(got[i], frames[i].pose), i
    icp.engine.close()
    # apps/pairwise_main.cpp: the known-answer benchmark, all three solvers + the closed-form row
    import re
    exe2 = os.path.join(build_dir, "pairwise_hostemu")
    subprocess.run(["/usr/bin/g++", "-O2", "-std=c++11", "-o", exe2, os.path.join(ROOT, "apps", "pairwise_main.cpp"), "-L" + build_dir,
                    "-lmvicp_hostemu", "-Wl,-rpath," + build_dir], check=True)
    A._write_cloud(tmp_path / "c.xyz", sc["pts"][0], sc["nor"][0])
    for extra in ([], ["--pointToPlane"]):
        r = subprocess.run([exe2, f"--cloud={tmp_path}/c.xyz"] + extra, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr
        m = re.findall(r"diff_tra:([0-9.e+-]+)\t diff_rot_degrees:([0-9.e+-]+)", r.stdout)
        assert len(m) == 4 and all(float(a) < 1e-8 and float(b) < 1e-4 for a, b in m[1:]) and (extra or float(m[0][0]) < 1e-12)


@pytest.mark.parametrize("xflags", [8, 16, 25, 32], ids=["no-adjacency", "no-obb", "no-adj-no-obb-no-seed", "step-loop"])
def test_schedules_are_bit_identical(emu, oracle, golden_dir, xflags):
    """Default: far rounds (no seeds yet / first seeded round) test the internal nodes against hybrid oriented boxes (csrc/far.cuh).
    MVICP_FLAG_NO_OBB: axis-aligned boxes only.  Same matches, same distances, same poses -- over ICP rounds that go from far to
    converged, on fp32 and fp64 storage, with exact duplicates (ties -> lowest index) and with tiny clouds."""
    from helpers import scene
    from mv_lm_icp_b200 import Engine, synth
    XF = xflags
    sc = scene(4, 3001, 27)
    edges = synth.ring_edges(4, 2)
    runs = []
    for flags in (0, XF):
        eng = Engine(flags=flags); eng.set_frames(sc["pts"], sc["nor"]); eng.set_graph(edges); eng.set_poses(sc["poses_init"])
        out = []
        for rnd in range(6 if emu.order == "ascending" else 3):
            s = eng.icp_round(0.05, 2, 1, True)
            out.append((eng.get_poses(), s["num_iterations"], [eng.get_nn(e) for e in range(len(edges)) if edges[e][0] != 0]))
        runs.append(out); eng.close()
    for (P0, it0, nn0), (P1, it1, nn1) in zip(*runs):
        assert it0 == it1 and np.array_equal(P0.view(np.uint64), P1.view(np.uint64))
        for (i0, d0), (i1, d1) in zip(nn0, nn1):
            assert np.array_equal(i0, i1) and np.array_equal(d0.view(np.uint64), d1.view(np.uint64))
    # fp64 storage, non-rigid poses, real scan (quantised coordinates): three slightly different poses, seeded
    g = np.load(f"{golden_dir}/bunny_pair.npz")
    res = []
    for flags in (0, XF):
        eng = Engine(flags=flags); eng.set_frames([g["pts0"], g["pts1"]], [g["nor0"], g["nor1"]]); eng.set_graph([(1, 0)])
        out = []
        for k in range(3):
            P1 = g["pose1"].copy(); P1[:3, 3] += 2e-4 * k
            eng.set_poses([g["pose0"], P1]); eng.correspond(0.05); out.append(eng.get_nn(0))
        res.append(out); eng.close()
    assert np.array_equal(res[0][0][0], g["nn_idx"])
    for (i0, d0), (i1, d1) in zip(*res):
        assert np.array_equal(i0, i1) and np.array_equal(d0.view(np.uint64), d1.view(np.uint64))
    # exact duplicates (distance ties -> lowest index) and clouds with fewer than ten points (no certificate possible)
    rng = np.random.default_rng(2)
    a = (rng.normal(size=(400, 3)) * 0.01).astype(np.float32).astype(np.float64); a[100:140] = a[0:40]
    b = a[::3] + np.float32(1e-4); tiny = a[:7].copy()
    res = []
    for flags in (0, XF):
        eng = Engine(flags=flags); eng.set_frames([a, b.astype(np.float32).astype(np.float64), tiny], None); eng.set_graph([(1, 0), (1, 2), (2, 0)])
        eng.set_poses([np.eye(4)] * 3, [1, 0, 0])
        out = []
        for k in range(3):
            eng.correspond(0.05); out.append([eng.get_nn(e) for e in range(3)])
        res.append(out); eng.close()
    for r0, r1 in zip(*res):
        for (i0, d0), (i1, d1) in zip(r0, r1):
            assert np.array_equal(i0, i1) and np.array_equal(d0.view(np.uint64), d1.view(np.uint64))


def test_closed_form_pairwise(emu, oracle):
    import test_gpu_zz_closed_form as T
    for n in (1, 3, 300, 20011):
        T.test_point_to_point_matches_oracle(oracle, n)
    T.test_reflection_branch_follows_the_reference(oracle)
    for n in (300, 20011):
        T.test_point_to_plane_matches_oracle(oracle, n)
    T.test_arguments()


def test_every_kernel_family_under_address_sanitizer(tmp_path):
    """tools/sanitize_run.py (every kernel family, both storage modes, general path, 40 views, experimental schedules) + the
    closed forms on an AddressSanitizer build of the emulated engine: device buffers are heap blocks there, so an out-of-bounds
    access by a kernel aborts the run (the CPU counterpart of profiles/r1_sanitizer.txt's memcheck)."""
    import subprocess
    import build_hostemu
    so = build_hostemu.build(asan=True)
    asan = subprocess.run(["/usr/bin/g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    script = tmp_path / "run.py"
    script.write_text(f"""
import sys, ctypes as C, runpy
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, 'tests')!r})
from mv_lm_icp_b200 import _lib, ICP_Ceres
lib = C.CDLL({so!r}); lib.mvicp_last_error.restype = C.c_char_p; _lib._lib = lib
runpy.run_path({os.path.join(ROOT, 'tools', 'sanitize_run.py')!r}, run_name='__main__')
from helpers import scene
sc = scene(2, 3001, 13)
ICP_Ceres.closed_form(sc['pts'][0], sc['pts'][0] + 0.01); ICP_Ceres.closed_form(sc['pts'][0], sc['pts'][0] + 0.01, sc['nor'][0])
print('ASAN RUN DONE')
""")
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0")
    r = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=1200, env=env)
    assert r.returncode == 0 and "ASAN RUN DONE" in r.stdout and "AddressSanitizer" not in r.stderr, r.stderr[-3000:]
