"""The public inputs of include/mvicp.h that the reference's drivers always pass with one value, checked against the CPU oracle:
fixed frames other than frame 0 (column map, gather lists, skyline envelope, shared vs global factor, write-back), every field of
mvicp_lm_options and every MVICP_TERM_* outcome, a robust edge of weight 0, mvicp_knn_self / mvicp_recompute_normals at every k,
fixed flags that change while certificates and the guessed median select are live, and a sharded run with a fixed middle frame.

Every case ends on decisions that are well clear of rounding (a trust-region radius that drops by orders of magnitude, a tolerance
met by a wide margin, an exactly singular block, an exactly NaN cost), so the engine and the oracle must agree on the termination
and the iteration counts, not only on the poses.  The check_* functions take their sizes as arguments:
tests/test_hostemu_engine.py runs them at small sizes on the CPU model of the engine."""
import ctypes as C
import os

import numpy as np
import pytest

from helpers import pose_rel_err, scene
from mv_lm_icp_b200 import COST_MIXED, COST_P2P, COST_P2PLANE, PARAM_AA, PARAM_QUAT, PARAM_SE3, Engine, synth
from mv_lm_icp_b200._lib import MvicpError
from mv_lm_icp_b200.api import FLAG_NO_CERT, FLAG_NO_SELECT_GUESS, TERMINATION, default_options

pytestmark = pytest.mark.gpu
TIGHT_TOL = 1e-8        # poses: what identical algorithms in fp64 reach (test_gpu_lm.py)
COST_TOL = 1e-9         # initial / final cost, relative
FIXED_TOL = 1e-14       # a fixed frame only goes through the parameter round trip
MVICP_ERR_INVALID = 1
EMPTY = (np.zeros(0, np.int32), np.zeros(0, np.int32))


# ---- shared plumbing ------------------------------------------------------------------------------------------------------
def _oracle_corr(O, pts, poses, edges, fixed, thresh=0.05):
    """Restated computeClosestPoints with a fixed mask: an edge whose src is fixed has no correspondences (frame.cpp:93).
    Returns (corr, weights, per-edge reference dicts or None)."""
    idxs, corr, w, ref = {}, [], [], []
    for s, d in edges:
        if fixed[s]:
            corr.append(EMPTY); w.append(np.float32(0)); ref.append(None); continue
        if d not in idxs:
            idxs[d] = O.KdIndex(pts[d], "kd")
        i, d2 = idxs[d].closest_points(pts[s], poses[s], poses[d], threads=8)
        f, sec, dist, ww, med = O.filter_edge(i, d2, np.float32(thresh))
        corr.append((f, sec)); w.append(ww); ref.append(dict(first=f, second=sec, weight=ww, nn_idx=i, nn_d2=d2))
    return corr, w, ref


def _assert_same_solve(summ, sref, P, Pref, ctx):
    assert TERMINATION[summ["termination"]] == TERMINATION[sref["termination"]], ctx
    assert summ["num_iterations"] == sref["num_iterations"], (ctx, summ, sref)
    assert summ["num_successful_steps"] == sref["num_successful_steps"], (ctx, summ, sref)
    assert abs(summ["initial_cost"] - sref["initial_cost"]) <= COST_TOL * sref["initial_cost"], ctx
    assert abs(summ["final_cost"] - sref["final_cost"]) <= COST_TOL * sref["final_cost"], ctx
    err = pose_rel_err(P, Pref)
    assert err <= TIGHT_TOL, (ctx, err)


def _solve_both(O, sc, poses, edges, corr, w, param, cost, robust=True, options=None, oracle_options=None, fixed=None, eng=None):
    """Feeds `corr` through mvicp_set_edge and solves on the engine and on the oracle from the same poses and fixed mask."""
    own = eng is None
    if own:
        eng = Engine(); eng.set_frames(sc["pts"], sc["nor"]); eng.set_graph(edges)
    eng.set_poses(poses, fixed)
    for e, (f, s) in enumerate(corr):
        eng.set_edge(e, f, s, w[e])
    summ = eng.optimize(param, cost, robust, options)
    P = eng.get_poses()
    if own:
        eng.close()
    Pref, sref, _ = O.optimize(sc["pts"], sc["nor"], poses, edges, corr, w, param=param, cost=cost, robust=robust,
                               se3_autodiff=True, threads=8, options=oracle_options, fixed=fixed)
    return summ, P, sref, Pref


# ---- 1. fixed frames anywhere ---------------------------------------------------------------------------------------------
# six views on the ring graph (synth.ring_edges(6, 2)); "dst_only": frame 4 is fixed and has no outgoing edge, so it enters the
# problem only as the dst of (3, 4) and (5, 4); "frame0_free": frame 0 is passed as free and mvicp_optimize must fix it itself
MASKS = {"middle": [1, 0, 0, 1, 0, 0], "last": [1, 0, 0, 0, 0, 1], "all_but_one": [1, 1, 1, 1, 1, 0],
         "frame0_free": [0, 0, 1, 0, 0, 0], "dst_only": [1, 0, 0, 0, 1, 0]}


def _mask_graph(name, n_views=6):
    edges = synth.ring_edges(n_views, 2)
    if name == "dst_only":
        edges = [(s, d) for s, d in edges if s != 4]
    return edges


def check_fixed_frames(O, mask, param, cost, n_points=2000):
    sc = scene(6, n_points, 7)
    fixed = MASKS[mask]
    edges = _mask_graph(mask)
    poses = sc["poses_init"]
    corr, w, ref = _oracle_corr(O, sc["pts"], poses, edges, fixed)
    eng = Engine(); eng.set_frames(sc["pts"], sc["nor"]); eng.set_graph(edges); eng.set_poses(poses, fixed)
    eng.correspond(0.05)
    for e, (s, d) in enumerate(edges):
        if fixed[s]:       # fixed before the first correspond: never searched
            assert eng.get_edge(e, arrays=False) == (0, np.float32(0)), (mask, e)
        else:
            f, sec, dist, ww = eng.get_edge(e)
            assert np.array_equal(f, ref[e]["first"]) and np.array_equal(sec, ref[e]["second"]) and ww == ref[e]["weight"], (mask, e)
    summ, P, sref, Pref = _solve_both(O, sc, poses, edges, corr, w, param, cost, fixed=fixed, eng=eng)
    eng.close()
    _assert_same_solve(summ, sref, P, Pref, (mask, param, cost))
    assert summ["num_successful_steps"] > 0
    for f in range(6):
        moved = np.max(np.abs(P[f] - poses[f]))
        if fixed[f] or f == 0:
            assert moved <= FIXED_TOL, (mask, f, moved)
        else:
            assert moved > 1e-6, (mask, f, moved)      # a free frame is really optimised
    # no damping at all (no Jacobi scaling, zero LM diagonal): a column left for a fixed frame would be an exactly singular block
    a, b = _options({"jacobi_scaling": 0, "min_lm_diagonal": 0.0})
    summ, P, sref, Pref = _solve_both(O, sc, poses, edges, corr, w, param, cost, options=a, oracle_options=b, fixed=fixed)
    _assert_same_solve(summ, sref, P, Pref, (mask, param, cost, "undamped"))
    assert TERMINATION[summ["termination"]] != "INVALID_STEPS"


@pytest.mark.parametrize("mask", list(MASKS))
@pytest.mark.parametrize("param", [PARAM_AA, PARAM_QUAT, PARAM_SE3])
@pytest.mark.parametrize("cost", [COST_P2P, COST_P2PLANE, COST_MIXED])
def test_fixed_frames_match_oracle(oracle, mask, param, cost):
    check_fixed_frames(oracle, mask, param, cost)


def _factor_bytes(M, edges, fixed):
    """Dynamic shared memory the LM step kernel would need with the factor inside: the skyline of the Cholesky factor (row r keeps
    columns rfirst[r]..r) plus the right-hand side and three work vectors, as mvicp_optimize lays them out (csrc/mvicp.cu)."""
    col, n = [-1] * M, 0
    for f in range(M):
        if not fixed[f] and f != 0:
            col[f] = n; n += 6
    rfirst = [(r // 6) * 6 for r in range(n)]
    for s, k in edges:
        if col[s] < 0 or col[k] < 0:
            continue
        for a, b in ((s, k), (k, s)):
            for i in range(6):
                rfirst[col[a] + i] = min(rfirst[col[a] + i], col[b])
    return 8 * (sum(r - rfirst[r] + 1 for r in range(n)) + n) + 8 * 3 * (n + 1)


SMEM_LIMIT = 220 * 1024


def check_factor_crosses_shared_memory(O, n_points=800):
    """The skyline factor of a ring of views is a narrow band (29 or 40 views: under 30 KB), so it stays in shared memory however
    many frames are fixed.  Here every frame is also linked to frame 1, the first free column, so every row of the factor is full:
    39 free frames (234 unknowns) need more than the 220 KB the step kernel may use and the factor lives in global memory; fixing
    one middle frame (228 unknowns) brings it back into shared memory, and freeing that frame again moves it out.  Three solves on
    one engine, each the oracle's."""
    M = 40
    sc = scene(M, n_points, 41)
    edges = sorted(set(synth.ring_edges(M, 2)) | {(f, 1) for f in range(3, M)})
    free = [1] + [0] * (M - 1)
    one = list(free); one[20] = 1
    assert _factor_bytes(M, edges, free) > SMEM_LIMIT >= _factor_bytes(M, edges, one)
    eng = Engine(); eng.set_frames(sc["pts"], sc["nor"]); eng.set_graph(edges)
    poses = sc["poses_init"]
    for fixed in (free, one, free):
        corr, w, _ = _oracle_corr(O, sc["pts"], poses, edges, fixed)
        summ, P, sref, Pref = _solve_both(O, sc, poses, edges, corr, w, PARAM_SE3, COST_P2PLANE, fixed=fixed, eng=eng)
        _assert_same_solve(summ, sref, P, Pref, fixed)
        assert np.max(np.abs(P[20] - poses[20])) <= FIXED_TOL if fixed[20] else np.max(np.abs(P[20] - poses[20])) > 1e-6
        poses = Pref
    eng.close()


def test_factor_crosses_shared_memory_limit(oracle):
    check_factor_crosses_shared_memory(oracle)


# ---- 2. solver options and every termination ------------------------------------------------------------------------------
# (name, option mutations, problem, expected termination).  Problems: "base" = four views, oracle correspondences; "zero_block" =
# the same with every edge of frame 2 (as src and as dst) given no correspondence, so frame 2's 6x6 block of the normal matrix is
# exactly zero; "weight0" = the base problem with edge (1, 0)'s weight set to 0 (SoftLOneLoss(0): NaN cost).
OPTION_SETS = [
    ("defaults", {}, "base", "FUNCTION_TOLERANCE"),
    ("no_jacobi_scaling", {"jacobi_scaling": 0}, "base", "FUNCTION_TOLERANCE"),
    ("gradient_tolerance", {"gradient_tolerance": 1e-2}, "base", "GRADIENT_TOLERANCE"),
    ("parameter_tolerance", {"parameter_tolerance": 1e-2}, "base", "PARAMETER_TOLERANCE"),
    ("three_iterations", {"max_num_iterations": 3, "function_tolerance": 0.0}, "base", "MAX_ITERATIONS"),
    # every step rejected (rho is about 1, never 10): the radius falls 1e4 -> 5e3 -> 1.25e3 -> 1.6e2, below 1e3 on step 3
    ("min_radius", {"min_relative_decrease": 10.0, "min_trust_region_radius": 1e3}, "base", "MIN_RADIUS"),
    ("strict_decrease", {"min_relative_decrease": 0.9}, "base", None),
    # a step of about the radius, six orders of magnitude below parameter_tolerance * |x|
    ("tiny_initial_radius", {"initial_trust_region_radius": 1e-14}, "base", "PARAMETER_TOLERANCE"),
    ("heavy_damping", {"min_lm_diagonal": 1e3}, "base", None),
    # the clamp on the LM diagonal applies to the scaled diagonal (at most 1 with Jacobi scaling, H_jj without): three steps of
    # different damping, so unscaled and scaled runs end at different poses
    ("heavy_damping_unscaled", {"jacobi_scaling": 0, "min_lm_diagonal": 1e3, "max_num_iterations": 3, "function_tolerance": 0.0},
     "base", "MAX_ITERATIONS"),
    ("capped_damping", {"max_lm_diagonal": 1e-8}, "base", None),
    ("huge_radius_no_diagonal", {"initial_trust_region_radius": 1e30, "max_trust_region_radius": 1e30, "min_lm_diagonal": 0.0},
     "base", None),
    # singular block, nothing to regularise it: the factorisation fails on the first step
    ("singular_one_invalid", {"max_num_consecutive_invalid_steps": 1, "jacobi_scaling": 0, "min_lm_diagonal": 0.0}, "zero_block",
     "INVALID_STEPS"),
    ("singular_five_invalid", {"max_num_consecutive_invalid_steps": 5, "jacobi_scaling": 0, "min_lm_diagonal": 0.0}, "zero_block",
     "INVALID_STEPS"),
    # the zero block's LM diagonal is min_lm_diagonal / radius = 1e-300 / radius: 0 (factorisation fails) while the radius is
    # above about 4e23, a subnormal (valid step) below.  From 1e24: invalid, invalid, valid; the successful steps then triple the
    # radius until it is above 4e23 again.  The invalid counter must restart after every valid step, or the third invalid step
    # in a row that never was ends the solve.
    ("invalid_counter_resets", {"max_num_consecutive_invalid_steps": 3, "jacobi_scaling": 0, "min_lm_diagonal": 1e-300,
                                "initial_trust_region_radius": 1e24, "max_trust_region_radius": 1e30}, "zero_block", None),
    ("weight0_robust", {}, "weight0", "EVAL_FAILURE"),
]


def _options(mut):
    """The same mutations on the engine's mvicp_lm_options and on the oracle's LmOptions (both start from the defaults)."""
    import oracle.oracle as O
    a, b = default_options(), O.default_options()
    for k, v in mut.items():
        setattr(a, k, v); setattr(b, k, v)
    return a, b


def _option_problem(O, problem, n_points):
    sc = scene(4, n_points, 7)
    edges = synth.ring_edges(4, 2)
    fixed = [1, 0, 0, 0]
    corr, w, _ = _oracle_corr(O, sc["pts"], sc["poses_init"], edges, fixed)
    if problem == "zero_block":
        for e, (s, d) in enumerate(edges):
            if 2 in (s, d):
                corr[e] = EMPTY; w[e] = np.float32(0)
    elif problem == "weight0":
        e = edges.index((1, 0)); w[e] = np.float32(0)
    return sc, edges, corr, w


def check_option_set(O, name, param, n_points=3000):
    _, mut, problem, want = next(s for s in OPTION_SETS if s[0] == name)
    sc, edges, corr, w = _option_problem(O, problem, n_points)
    a, b = _options(mut)
    summ, P, sref, Pref = _solve_both(O, sc, sc["poses_init"], edges, corr, w, param, COST_P2PLANE, options=a, oracle_options=b)
    if want is not None:
        assert TERMINATION[sref["termination"]] == want, (name, sref)        # the case tests what it says it tests
    if TERMINATION[sref["termination"]] == "EVAL_FAILURE":
        assert TERMINATION[summ["termination"]] == "EVAL_FAILURE" and summ["num_iterations"] == sref["num_iterations"] == 0
        assert summ["num_successful_steps"] == sref["num_successful_steps"] == 0
        assert np.max(np.abs(P - sc["poses_init"])) <= FIXED_TOL and np.max(np.abs(Pref - sc["poses_init"])) <= FIXED_TOL
        return summ
    _assert_same_solve(summ, sref, P, Pref, name)
    if name == "invalid_counter_resets":     # the pattern the comment above describes really happened
        assert summ["num_successful_steps"] >= 2 and summ["num_iterations"] - summ["num_successful_steps"] >= 3, summ
        assert TERMINATION[summ["termination"]] != "INVALID_STEPS", summ
    if name == "singular_five_invalid":
        assert summ["num_iterations"] == 5 and summ["num_successful_steps"] == 0, summ
    return summ


def test_option_table_reaches_every_termination():
    want = {s[3] for s in OPTION_SETS if s[3] is not None}
    assert want == set(TERMINATION), set(TERMINATION) - want
    assert len({s[0] for s in OPTION_SETS}) == len(OPTION_SETS)


@pytest.mark.parametrize("name", [s[0] for s in OPTION_SETS])
@pytest.mark.parametrize("param", [PARAM_AA, PARAM_SE3])
def test_option_set_matches_oracle(oracle, name, param):
    check_option_set(oracle, name, param)


def check_options_general_path(O, golden_dir, param=PARAM_SE3):
    """The Bunny scans with their own (non-rigid) sample poses run the general frame model; a reduced-iteration, unscaled,
    strict-decrease option set there."""
    g = np.load(f"{golden_dir}/bunny_pair.npz")
    pts = [g["pts0"], g["pts1"]]; nor = [g["nor0"], g["nor1"]]
    poses = np.stack([g["pose0"], g["pose1"]])
    edges = [(1, 0)]
    corr, w, _ = _oracle_corr(O, pts, poses, edges, [1, 0])
    a, b = _options({"jacobi_scaling": 0, "min_relative_decrease": 0.5, "max_num_iterations": 6})
    sc = {"pts": pts, "nor": nor}
    summ, P, sref, Pref = _solve_both(O, sc, poses, edges, corr, w, param, COST_P2PLANE, options=a, oracle_options=b)
    _assert_same_solve(summ, sref, P, Pref, "general")


def test_options_on_the_general_path(oracle, golden_dir):
    check_options_general_path(oracle, golden_dir)


# ---- 3. weight 0 through the real pipeline --------------------------------------------------------------------------------
def check_weight0_pipeline(O, n_points=3000):
    """Frame 2 is an exact copy of frame 0 at the same pose: every match of edge (2, 0) is at distance 0, the median is 0 and
    the weight is 0.  With the robust loss SoftLOneLoss(0) makes the cost NaN and the solve fails before its first step, poses
    unchanged; without the loss the same scene solves normally."""
    sc0 = scene(2, n_points, 7)
    sc = {"pts": [sc0["pts"][0], sc0["pts"][1], sc0["pts"][0].copy()], "nor": [sc0["nor"][0], sc0["nor"][1], sc0["nor"][0].copy()]}
    # in frame 0's coordinates, so that the transform between frames 2 and 0 is exactly the identity and every d^2 exactly 0
    P1 = np.linalg.solve(sc0["poses_init"][0], sc0["poses_init"][1]); P1[3] = [0, 0, 0, 1]
    poses = np.stack([np.eye(4), P1, np.eye(4)])
    edges = [(1, 0), (1, 2), (2, 0), (2, 1)]
    fixed = [1, 0, 0]
    eng = Engine(); eng.set_frames(sc["pts"], sc["nor"]); eng.set_graph(edges); eng.set_poses(poses)
    eng.correspond(0.05)
    corr, w, ref = _oracle_corr(O, sc["pts"], poses, edges, fixed)
    e20 = edges.index((2, 0))
    assert w[e20] == 0 and not np.any(ref[e20]["nn_d2"])
    for e in range(len(edges)):
        f, s, d, ww = eng.get_edge(e)
        assert np.array_equal(f, ref[e]["first"]) and np.array_equal(s, ref[e]["second"])
        assert np.float32(ww).view(np.uint32) == np.float32(ref[e]["weight"]).view(np.uint32), e
    summ = eng.optimize(PARAM_SE3, COST_P2PLANE, True)
    P = eng.get_poses()
    Pref, sref, _ = O.optimize(sc["pts"], sc["nor"], poses, edges, corr, w, param=PARAM_SE3, cost=COST_P2PLANE, robust=True,
                               threads=8)
    assert TERMINATION[summ["termination"]] == TERMINATION[sref["termination"]] == "EVAL_FAILURE"
    assert summ["num_iterations"] == sref["num_iterations"] == 0
    assert np.max(np.abs(P - poses)) <= FIXED_TOL and np.max(np.abs(Pref - poses)) <= FIXED_TOL
    eng.set_poses(poses)
    summ = eng.optimize(PARAM_SE3, COST_P2PLANE, False)
    P = eng.get_poses()
    eng.close()
    Pref, sref, _ = O.optimize(sc["pts"], sc["nor"], poses, edges, corr, w, param=PARAM_SE3, cost=COST_P2PLANE, robust=False,
                               threads=8)
    _assert_same_solve(summ, sref, P, Pref, "no loss")
    assert summ["num_successful_steps"] > 0 and TERMINATION[summ["termination"]] != "EVAL_FAILURE"


def test_weight0_edge_through_the_pipeline(oracle):
    check_weight0_pipeline(oracle)


# ---- 4. knn_self and normals at every k -----------------------------------------------------------------------------------
KS = (1, 2, 3, 9, 10, 11, 15, 16)


def _brute_knn(P, rows, k):
    """k nearest of each row's point in its own cloud, the point included: (dx*dx + dy*dy) + dz*dz in fp64, ordered by
    (d^2, index); -1 where the cloud has fewer than k points."""
    out = np.full((len(rows), k), -1, np.int32)
    idx = np.arange(len(P))
    for r, i in enumerate(rows):
        d = P - P[i]
        d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        o = np.lexsort((idx, d2))[:k]
        out[r, :len(o)] = o
    return out


def _knn_clouds(f32, big):
    """Named clouds: tiny ones (n = 1, 2 and around every k), sizes around the 8-point leaf, a lattice whose spacing is a power
    of two (exact ties at many distances, the k-th included), a cloud of exact duplicates, and a large jittered cloud."""
    rng = np.random.default_rng(11 if f32 else 12)
    sizes = sorted({1, 2} | {n for k in KS for n in (k - 1, k, k + 1) if n > 0} | {7, 8, 9, 23, 24, 25})
    clouds = [(f"n{n}", rng.normal(size=(n, 3)) * 0.02) for n in sizes]
    g = np.arange(6) * 2.0 ** -6
    clouds.append(("lattice", np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3) + 0.25))
    base = rng.normal(size=(150, 3)) * 0.01
    clouds.append(("duplicates", np.concatenate([base, base[::-1], base[:40]])))
    if big:
        clouds.append(("big", rng.normal(size=(big, 3)) * [0.05, 0.05, 0.01]))
    if f32:
        clouds = [(nm, c.astype(np.float32).astype(np.float64)) for nm, c in clouds]
    return clouds


@pytest.mark.parametrize("f32", [True, False], ids=["fp32-exact", "fp64"])
def test_knn_self_every_k(f32):
    check_knn_self(f32)


def check_knn_self(f32, big=30011, ks=KS, sample=300):
    clouds = _knn_clouds(f32, big)
    # frame 0 is a cloud of its own, so every named cloud is a frame other than 0 (storage is per engine: fp32 only if every
    # coordinate of every frame is fp32-exact)
    pts = [np.random.default_rng(3).normal(size=(40, 3)) * 0.02] + [c for _, c in clouds]
    if f32:
        pts[0] = pts[0].astype(np.float32).astype(np.float64)
    eng = Engine(); eng.set_frames(pts)
    rng = np.random.default_rng(4)
    for f, (name, P) in enumerate(clouds, start=1):
        rows = np.arange(len(P)) if len(P) <= 2000 else np.sort(rng.choice(len(P), sample, replace=False))
        for k in ks:
            got = eng.knn_self(f, k)
            assert got.shape == (len(P), k)
            want = _brute_knn(P, rows, k)
            bad = np.nonzero(np.any(got[rows] != want, axis=1))[0]
            assert len(bad) == 0, (name, k, rows[bad[:3]], got[rows[bad[:3]]], want[bad[:3]])
            if len(P) < k:
                assert np.all(got[:, len(P):] == -1)
    # a lattice has ties at the k-th distance: confirm the cloud tests what it claims
    lat = next(c for nm, c in clouds if nm == "lattice")
    d = np.sort(np.sum((lat - lat[0]) ** 2, axis=1))
    assert any(d[k - 1] == d[k] for k in ks)
    # argument checks: k outside [1, KNN_MAXK = 16], a frame out of range
    buf = np.zeros(17 * 64, np.int32)
    for frame, k in ((1, 0), (1, 17), (-1, 3), (len(pts), 3)):
        rc = eng._l.mvicp_knn_self(eng._ctx, C.c_int32(frame), C.c_int32(k), buf.ctypes.data_as(C.POINTER(C.c_int32)))
        assert rc == MVICP_ERR_INVALID, (frame, k, rc)
    for k in (2, 17):       # pointSetPCA needs 3 neighbours; the k-best list holds 16
        with pytest.raises(MvicpError) as ex:
            eng.recompute_normals(k)
        assert ex.value.code == MVICP_ERR_INVALID
    eng.close()


def check_normals_every_k(O, n_points=5000, ks=(3, 16)):
    """mvicp_recompute_normals against the oracle at the smallest and the largest k, on the points whose k nearest neighbours are
    unique (no tie at the k-th distance) and whose smallest eigenvalue is separated (the filter of
    test_gpu_normals.py::test_normals_real_scan_and_lm_uses_them).  A frame with fewer than k points: every point's neighbour list is
    the whole cloud, so every point gets the normal of the whole cloud, as in the oracle; a one-point frame has a zero covariance,
    and both sides return the first axis (1, 0, 0)."""
    sc = scene(2, n_points, 21)
    few = np.random.default_rng(6).normal(size=(9, 3)) * [0.03, 0.02, 0.01]
    pts = [sc["pts"][0], sc["pts"][1], few, few[:1].copy()]
    eng = Engine(); eng.set_frames(pts)
    for k in ks:
        nor, _ = eng.recompute_normals(k)
        for f in (0, 1):
            ref, nn = O.recompute_normals(pts[f], k, threads=8, want_nn=True)
            sel = np.arange(0, len(pts[f]), 5)
            nxt = _brute_knn(pts[f], sel, k + 1)
            d2 = [np.sum((pts[f][nxt[:, j]] - pts[f][sel]) ** 2, axis=1) for j in (k - 1, k)]
            sel = sel[d2[0] != d2[1]]
            Q = pts[f][nn[sel]]; Cn = Q - Q.mean(1, keepdims=True)
            wv = np.linalg.eigvalsh(np.einsum("nki,nkj->nij", Cn, Cn))
            sel = sel[(wv[:, 1] - wv[:, 0]) > 1e-3 * wv[:, 2]]
            assert len(sel) > len(pts[f]) // 10, (k, f, len(sel))
            assert np.max(np.abs(nor[f][sel] - ref[sel])) < 1e-9, (k, f)
            assert np.all(nor[f][:, 2] <= 0) and np.max(np.abs(np.linalg.norm(nor[f], axis=1) - 1)) < 1e-12
        if k > len(few):
            ref = O.recompute_normals(few, k)
            assert np.max(np.abs(nor[2] - ref)) < 1e-12 and np.max(np.abs(nor[2] - nor[2][0])) < 1e-12, k
            assert np.array_equal(eng.knn_self(2, k)[:, len(few):], np.full((len(few), k - len(few)), -1, np.int32))
        assert np.array_equal(nor[3], [[1.0, 0.0, 0.0]]) and np.array_equal(O.recompute_normals(pts[3], k), [[1.0, 0.0, 0.0]]), k
    eng.close()


def test_normals_at_k3_and_k16(oracle):
    check_normals_every_k(oracle)


# ---- 5. fixed flags that change in converged rounds -----------------------------------------------------------------------
def check_fixed_toggle_in_converged_rounds(O, n_views=5, n_points=5003, warm=8):
    """Full solves until converged, then rounds that keep certified matches and guess the median (max_num_iterations = 0 or 1,
    test_gpu_corr.py::test_certified_matches_are_exact).  Frame 2 is fixed for some of those rounds -- its edges are then not searched,
    and a full solve moves its neighbours -- and freed again: its edges come back with matches, certificates and a median window from
    an older round.  Every round must give the matches of an engine that searches every query and always runs the full select."""
    sc = scene(n_views, n_points, 21)
    edges = synth.ring_edges(n_views, 2)
    one = default_options(); one.max_num_iterations = 1
    none = default_options(); none.max_num_iterations = 0
    # (frame 2 fixed, options of the solve that ends the round)
    schedule = [(0, none), (0, none), (1, None), (1, none), (0, none), (0, none), (0, none), (1, one), (0, none), (0, none)]
    engs = [Engine(flags=f) for f in (0, FLAG_NO_CERT | FLAG_NO_SELECT_GUESS)]
    for eng in engs:
        eng.set_frames(sc["pts"], sc["nor"]); eng.set_graph(edges); eng.set_poses(sc["poses_init"])
        for _ in range(warm):
            eng.correspond(0.05); eng.optimize()
    refree = schedule.index((0, none), 3)
    for rnd, (fx2, opt) in enumerate(schedule):
        if rnd == refree:
            before = engs[0].stats()
        fixed = [1] + [0] * (n_views - 1); fixed[2] = fx2
        out = []
        for eng in engs:
            poses = eng.get_poses()
            eng.set_poses(poses, fixed)     # the poses this engine handed out: only the flags change
            eng.correspond(0.05)
            out.append(([eng.get_nn(e) for e, (s, d) in enumerate(edges) if not fixed[s]],
                        [eng.get_edge(e, arrays=False) for e in range(len(edges))]))
            eng.optimize(options=opt)
        (nn0, meta0), (nn1, meta1) = out
        for (i0, d0), (i1, d1) in zip(nn0, nn1):
            assert np.array_equal(i0, i1) and np.array_equal(d0.view(np.uint64), d1.view(np.uint64)), rnd
        assert meta0 == meta1, rnd
        assert np.array_equal(engs[0].get_poses().view(np.uint64), engs[1].get_poses().view(np.uint64)), rnd
    after = engs[0].stats()
    assert after["cert_rounds"] > before["cert_rounds"] and after["cert_reused"] > before["cert_reused"], (before, after)
    assert after["select_guess_rounds"] > before["select_guess_rounds"], (before, after)
    assert engs[1].stats()["cert_rounds"] == 0 and engs[1].stats()["select_guess_rounds"] == 0
    # the last round against the oracle, from the poses it started from
    _, ref_w, ref = _oracle_corr(O, sc["pts"], poses, edges, fixed)
    for j, e in enumerate([e for e, (s, d) in enumerate(edges) if not fixed[s]]):
        i1, d1 = nn1[j]
        assert np.array_equal(i1, ref[e]["nn_idx"]) and np.array_equal(d1.view(np.uint64), ref[e]["nn_d2"].view(np.uint64)), e
        assert meta1[e] == (len(ref[e]["first"]), ref_w[e]), e
    # mvicp_set_edge replaces an edge's matches and voids the certificates; a fixed-flag change that follows must not revive them
    e1 = edges.index((1, 0))
    out = []
    fixed[2] ^= 1
    for eng in engs:
        eng.set_edge(e1, *EMPTY, 0.0)
        eng.optimize(options=none)
        poses = eng.get_poses(); eng.set_poses(poses, fixed); eng.correspond(0.05)
        out.append(eng.get_nn(e1))
    _, _, ref = _oracle_corr(O, sc["pts"], poses, edges, fixed)
    for i, d in out:
        assert np.array_equal(i, ref[e1]["nn_idx"]) and np.array_equal(d.view(np.uint64), ref[e1]["nn_d2"].view(np.uint64))
    for eng in engs:
        eng.close()


def test_fixed_toggle_in_converged_rounds(oracle):
    check_fixed_toggle_in_converged_rounds(oracle)


# ---- 6. sharded run with a fixed middle frame -----------------------------------------------------------------------------
SHARD_FIXED = [1, 0, 1, 0, 0, 0]


def _run_sharded(rank, world, port, out_dir, n_points, rounds):
    import torch
    import torch.distributed as dist
    import mv_lm_icp_b200 as mv
    from mv_lm_icp_b200.dist import broadcast_unique_id, edge_owners
    from test_gpu_multi import _scene_file
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    sc = _scene_file(out_dir, 6, n_points, 22)
    edges = synth.ring_edges(6, 2)
    eng = mv.Engine(device=rank)
    eng.set_frames(sc["pts"], sc["nor"]); eng.set_graph(edges)
    eng.comm_init(broadcast_unique_id(mv.nccl_unique_id, rank, device="cuda"), rank, world)
    eng.set_poses(sc["poses_init"], SHARD_FIXED)
    out = []
    for _ in range(rounds):
        s = eng.icp_round(0.05, mv.PARAM_SE3, mv.COST_P2PLANE, True)
        out.append((eng.get_poses(), s["num_iterations"]))
    own = edge_owners(edges, [len(p) for p in sc["pts"]], world, SHARD_FIXED)
    for e in range(len(edges)):
        try:
            eng.get_nn(e); mine = True
        except RuntimeError:
            mine = False
        assert mine == (own[e] == rank), (e, rank, own[e])
    np.save(os.path.join(out_dir, f"poses_{rank}.npy"), np.stack([o[0] for o in out]))
    np.save(os.path.join(out_dir, f"iters_{rank}.npy"), np.array([o[1] for o in out]))
    eng.close()
    dist.barrier(); dist.destroy_process_group()


def test_two_gpus_with_a_fixed_middle_frame(tmp_path):
    """fixed = [1, 0, 1, 0, 0, 0] before the first mvicp_correspond: the edges of frame 2 belong to no rank, the others are cut by
    query count (dist.edge_owners), and poses and iteration counts are bit-identical to the single-GPU run."""
    import torch
    import torch.multiprocessing as mp
    from test_gpu_multi import _free_port, _scene_file
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    n_points, rounds = 20011, 3
    sc = _scene_file(str(tmp_path), 6, n_points, 22)
    edges = synth.ring_edges(6, 2)
    eng = Engine(); eng.set_frames(sc["pts"], sc["nor"]); eng.set_graph(edges); eng.set_poses(sc["poses_init"], SHARD_FIXED)
    ref = []
    for _ in range(rounds):
        s = eng.icp_round(0.05, PARAM_SE3, COST_P2PLANE, True)
        ref.append((eng.get_poses(), s["num_iterations"]))
    eng.close()
    assert np.max(np.abs(ref[-1][0][2] - sc["poses_init"][2])) <= FIXED_TOL
    mp.spawn(_run_sharded, args=(2, _free_port(), str(tmp_path), n_points, rounds), nprocs=2, join=True)
    for r in range(2):
        P = np.load(tmp_path / f"poses_{r}.npy"); it = np.load(tmp_path / f"iters_{r}.npy")
        assert it.tolist() == [x[1] for x in ref]
        assert np.array_equal(P.view(np.uint64), np.stack([x[0] for x in ref]).view(np.uint64))
