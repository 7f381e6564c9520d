"""Pins the oracle's correspondence restatement (oracle_icp.cpp) against the reference's own nanoflann (its stored answers in
tests/golden/ref_pins.npz, and the library itself when oracle/_ref was built), against brute force, and against the committed
golden vectors."""
import hashlib

import numpy as np

from helpers import scene
from mv_lm_icp_b200 import synth


def _edge_inputs(n=4000, cfg=31):
    sc = scene(3, n, cfg)
    return sc, (1, 0)


def test_kd_restatement_equals_brute_force(oracle):
    sc, (s, d) = _edge_inputs()
    for poses in (sc["poses_init"], sc["poses_gt"]):
        a = oracle.KdIndex(sc["pts"][d], "kd").closest_points(sc["pts"][s], poses[s], poses[d], threads=4)
        b = oracle.KdIndex(sc["pts"][d], "brute").closest_points(sc["pts"][s], poses[s], poses[d], threads=4)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))


def test_restatement_equals_reference_nanoflann(oracle, golden_dir):
    sc, (s, d) = _edge_inputs(20000, 32)
    g = np.load(f"{golden_dir}/ref_pins.npz")
    for name in ("poses_init", "poses_gt"):   # the reference's answers, stored (tests/golden/make_golden.py:ref_pins)
        poses = sc[name]
        a = oracle.KdIndex(sc["pts"][d], "kd").closest_points(sc["pts"][s], poses[s], poses[d], threads=4)
        assert hashlib.sha256(a[1].tobytes()).hexdigest() == str(g[f"corr_{name}_d2_sha256"])   # minimal squared distance: bit-exact
        assert np.array_equal(a[0], g[f"corr_{name}_idx"])                                   # no exact ties on jittered data
    if oracle.ref_lib() is None:
        return
    ties = 0
    for poses in (sc["poses_init"], sc["poses_gt"]):
        a = oracle.KdIndex(sc["pts"][d], "kd").closest_points(sc["pts"][s], poses[s], poses[d], threads=4)
        r = oracle.KdIndex(sc["pts"][d], "ref").closest_points(sc["pts"][s], poses[s], poses[d], threads=4)
        assert np.array_equal(a[1].view(np.uint64), r[1].view(np.uint64))    # minimal squared distance: bit-exact
        ties += int((a[0] != r[0]).sum())                                     # index may differ only on exact ties
        same_d = a[1][a[0] != r[0]] == r[1][a[0] != r[0]]
        assert same_d.all()
    assert ties == 0   # none on jittered synthetic data (SURVEY section 7)


def test_golden_bunny_pair(oracle, golden_dir):
    """Golden = reference nanoflann on the reference's own scans (tests/golden/make_golden.py)."""
    g = np.load(f"{golden_dir}/bunny_pair.npz")
    idx, d2 = oracle.KdIndex(g["pts0"], "kd").closest_points(g["pts1"], g["pose1"], g["pose0"], threads=4)
    assert np.array_equal(d2.view(np.uint64), g["nn_d2"].view(np.uint64))
    assert np.array_equal(idx, g["nn_idx"])
    f, s, dist, w, med = oracle.filter_edge(idx, d2, np.float32(0.05))
    assert np.array_equal(f, g["first"]) and np.array_equal(s, g["second"]) and np.array_equal(dist, g["dist"])
    assert np.float32(w) == g["weight"] and med == g["median"]
    if oracle.ref_lib() is not None:
        ri, rd = oracle.KdIndex(g["pts0"], "ref").closest_points(g["pts1"], g["pose1"], g["pose0"])
        assert np.array_equal(ri, g["nn_idx"]) and np.array_equal(rd, g["nn_d2"])


def test_golden_dinosaur_pair(oracle, golden_dir):
    """The reference's second sample set (millimetre units, |x| up to 686, NN distances of tens of mm, 5-digit pose
    matrices): golden = reference nanoflann, cutoff 25 (tests/golden/make_golden.py:dino_pair)."""
    g = np.load(f"{golden_dir}/dino_pair.npz")
    idx, d2 = oracle.KdIndex(g["pts0"], "kd").closest_points(g["pts1"], g["pose1"], g["pose0"], threads=4)
    assert np.array_equal(d2.view(np.uint64), g["nn_d2"].view(np.uint64))
    assert np.array_equal(idx, g["nn_idx"])
    f, s, dist, w, med = oracle.filter_edge(idx, d2, np.float32(25.0))
    assert np.array_equal(f, g["first"]) and np.array_equal(s, g["second"]) and np.array_equal(dist, g["dist"])
    assert np.float32(w) == g["weight"] and med == g["median"] and 0 < len(f) < len(idx)
    if oracle.ref_lib() is not None:
        ri, rd = oracle.KdIndex(g["pts0"], "ref").closest_points(g["pts1"], g["pose1"], g["pose0"])
        assert np.array_equal(ri, g["nn_idx"]) and np.array_equal(rd, g["nn_d2"])


def test_filter_semantics(oracle):
    d2 = np.array([1e-6, 4e-6, 0.0025000001, 9e-6, 0.0024, 1.0])     # sqrt: .001 .002 >.05 .003 .049 1
    idx = np.arange(6, dtype=np.int32)[::-1].copy()
    f, s, dist, w, med = oracle.filter_edge(idx, d2, np.float32(0.05))
    assert f.tolist() == [0, 1, 3, 4] and s.tolist() == [5, 4, 2, 1]
    assert med == np.sort(dist)[len(dist) // 2] == 0.003              # upper median (frame.cpp:166-168)
    assert w == np.float32(0.003 * 1.5)
    # threshold is the float 0.05f promoted to double, strict "<" (frame.cpp:156)
    thr = float(np.float32(0.05))
    f2, *_ = oracle.filter_edge(np.zeros(2, np.int32), np.array([thr, np.nextafter(thr, 0)]) ** 2, np.float32(0.05))
    assert len(f2) <= 1
    f3, s3, d3, w3, m3 = oracle.filter_edge(np.zeros(2, np.int32), np.array([1.0, 4.0]), np.float32(0.05))
    assert len(f3) == 0 and w3 == 0 and np.isnan(m3)                  # reference: UB; oracle: weight 0


def test_pose_graph_knn_is_the_ring(oracle):
    sc = scene(6, 20011, 22)
    nb = oracle.pose_graph_knn(sc["poses_gt"], 2)
    edges = [(i, int(j)) for i in range(6) for j in nb[i]]
    assert sorted(edges) == sorted(synth.ring_edges(6, 2))
    for i in range(6):
        assert set(nb[i].tolist()) == {(i - 1) % 6, (i + 1) % 6}


def test_knn_restatement_equals_reference_nanoflann(oracle, golden_dir):
    """Frame::getNeighbours (frame.cpp:208-242): the oracle's k-NN against the reference's nanoflann knnSearch on the
    reference's own scan.  Squared distances must agree bit for bit; indices may differ only inside groups of exactly
    equal distance (the scan's coordinates are quantised, so such ties exist; nanoflann orders them by traversal).  The
    reference's answers are stored (tests/golden/make_golden.py:ref_pins); the library is asked as well when oracle/_ref was built."""
    g = np.load(f"{golden_dir}/bunny_pair.npz")
    pts = g["pts0"]
    pins = np.load(f"{golden_dir}/ref_pins.npz")
    assert np.array_equal(pins["knn_query"], np.arange(0, len(pts), 53))
    kd = oracle.KdIndex(pts, "kd"); rf = oracle.KdIndex(pts, "ref") if oracle.ref_lib() is not None else None
    differing = 0
    for k, i in enumerate(pins["knn_query"]):
        a = oracle.knn(kd, pts[i], 10); b = (pins["knn_idx"][k], pins["knn_d2"][k])
        if rf is not None:
            live = oracle.knn(rf, pts[i], 10)
            assert np.array_equal(live[0], b[0]) and np.array_equal(live[1].view(np.uint64), b[1].view(np.uint64))
        assert np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))
        assert a[0][0] == i == b[0][0] and a[1][0] == 0.0            # the point itself comes first
        if not np.array_equal(a[0], b[0]):
            differing += 1
            for j in np.where(a[0] != b[0])[0]:                      # every disagreement sits in a tie group
                assert (a[1] == a[1][j]).sum() > 1 or np.sum((pts[b[0][j]] - pts[i]) ** 2) == a[1][-1]
    assert differing > 0    # documents that ties do occur on the real scans


def test_normals_restatement(oracle, golden_dir):
    """pointSetPCA (common.h:331-346) restated: unit eigenvector of the smallest eigenvalue of sum (p-c)(p-c)^T over the
    10 nearest neighbours, flipped to n.z <= 0 -- checked against numpy.linalg.eigh."""
    sc = scene(3, 4000, 31)
    pts = sc["pts"][1]
    nor, nn = oracle.recompute_normals(pts, 10, threads=4, want_nn=True)
    assert np.all(nor[:, 2] <= 0) and np.max(np.abs(np.linalg.norm(nor, axis=1) - 1)) < 1e-12
    P = pts[nn]; C = P - P.mean(1, keepdims=True)
    w, V = np.linalg.eigh(np.einsum("nki,nkj->nij", C, C))
    v = V[:, :, 0]; v = np.where(v[:, 2:3] > 0, -v, v)
    good = (w[:, 1] - w[:, 0]) > 1e-6 * w[:, 2]
    assert good.mean() > 0.99 and np.max(np.abs(v[good] - nor[good])) < 1e-7
    assert np.median(np.abs(np.sum(nor * sc["nor"][1], axis=1))) > 0.99     # and they are the surface normals
