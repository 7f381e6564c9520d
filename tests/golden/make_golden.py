"""Regenerates tests/golden/*.npz.  Run in the build container (needs /root/reference):  python tests/golden/make_golden.py

bunny_pair.npz   config 1 of BASELINE.json: the reference's own sample scans samples/Bunny_RealData/cloudXYZ_{0,1}.xyz
                 (x y z nx ny nz per line; the loader's trailing garbage point, common.h:224-239, is NOT reproduced)
                 with poses_{0,1}.txt (4x4 row-major).  Stored as float64 exactly as parsed.
                 + nn_idx / nn_d2: output of the REFERENCE's nanoflann (oracle/_ref/libref_nanoflann.so, compiled from
                 /root/reference/include/nanoflann.hpp) for edge 1 -> 0 under those poses, i.e. the pinned answer of
                 Frame::computeClosestPointsToNeighbours' inner loop (frame.cpp:129-138);
                 + first/second/dist/weight of frame.cpp:140-176 from those.
dino_pair.npz    the reference's second sample set, samples/dinosaur/cloud_{1,2}.xyz with pose_{1,2}.txt: millimetre units
                 (|coordinates| up to 686, NN distances of tens of mm), 5-digit pose matrices (not exactly orthonormal):
                 edge 2 -> 1, reference nanoflann answer + frame.cpp:140-176 at cutoff 25 (the default 0.05 m is meaningless
                 in mm); pins the fp32 screening bound at a different coordinate magnitude.
lm_golden.npz    oracle LM outputs (final poses, iteration trace) on a small seeded synthetic scene for every
                 parameterisation x cost; pins the oracle against accidental change (NOT against Ceres: unpinned).
bunny18.npz      the reference's DEFAULT multiview workload (main_multiview.cpp:33-36,63: --limit=40 --step=2 on Bunny_RealData): the 18
                 scans cloudXYZ_{0,2,..,34}.xyz (224 673 points; xyz only -- the default run recomputes the normals; stored as int32
                 units of 1e-8 m, which is lossless for the <= 8-decimal text: parsed double == int / 1e8 exactly) with poses_{0,2,..,34}.txt
                 (ground truth, non-rigid: singular values 1, 0.9957, 0.9957) and the initial poses of main_multiview.cpp:78-84
                 (frame 0 = GT, the others addNoise(GT, 0.02, 0.01), common.h:38-67; the reference's default-seeded mt19937 stream
                 is not reproduced -- same noise model, numpy seed 0xB18).  Used by `bench.py --config real` and tests/test_gpu_real18.py.
sophus_vectors.npz  the SE3 group elements / tangents of ext/sophus-ceres/test/core/test_se3.cpp:40-82 (values only).
ref_pins.npz     answers of the reference's own code (oracle/_ref) that tests/test_oracle_corr.py and tests/test_oracle_functor_pin.py
                 compare the oracle with, so that those comparisons run where the reference tree is absent:
                 corr_*: nanoflann's 1-NN for edge 1 -> 0 of synth.make_scene(3, 20000, 32) under poses_init / poses_gt (every
                 index, and the sha256 of the squared distances' bytes); knn_*: nanoflann's knnSearch(10) for every 53rd point of
                 bunny_pair.npz's pts0; gfun_* / pfun_* / quat_*: inputs and outputs of the reference functor text for the first
                 iterations of the seeded loops of test_oracle_functor_pin.py (a sample: the full loops would not fit in 1 MB).
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402
from mv_lm_icp_b200 import synth  # noqa: E402

REF = "/root/reference/samples/Bunny_RealData"
OUT = os.path.dirname(os.path.abspath(__file__))


def bunny_pair():
    c = [np.loadtxt(f"{REF}/cloudXYZ_{i}.xyz") for i in (0, 1)]
    P = [np.loadtxt(f"{REF}/poses_{i}.txt") for i in (0, 1)]
    ref = O.KdIndex(c[0][:, :3], "ref")
    idx, d2 = ref.closest_points(c[1][:, :3], P[1], P[0])
    first, second, dist, w, med = O.filter_edge(idx, d2, np.float32(0.05))
    np.savez_compressed(os.path.join(OUT, "bunny_pair.npz"), pts0=c[0][:, :3], nor0=c[0][:, 3:6], pts1=c[1][:, :3],
                        nor1=c[1][:, 3:6], pose0=P[0], pose1=P[1], nn_idx=idx, nn_d2=d2, first=first, second=second,
                        dist=dist, weight=w, median=med)
    print("bunny_pair:", c[0].shape, c[1].shape, "inliers", len(first), "weight", w)


def dino_pair():
    D = "/root/reference/samples/dinosaur"
    c = [np.loadtxt(f"{D}/cloud_{i}.xyz") for i in (1, 2)]
    P = [np.loadtxt(f"{D}/pose_{i}.txt") for i in (1, 2)]
    ref = O.KdIndex(c[0][:, :3], "ref")
    idx, d2 = ref.closest_points(c[1][:, :3], P[1], P[0])
    first, second, dist, w, med = O.filter_edge(idx, d2, np.float32(25.0))
    np.savez_compressed(os.path.join(OUT, "dino_pair.npz"), pts0=c[0][:, :3], nor0=c[0][:, 3:6], pts1=c[1][:, :3], nor1=c[1][:, 3:6],
                        pose0=P[0], pose1=P[1], nn_idx=idx, nn_d2=d2, first=first, second=second, dist=dist, weight=w, median=med)
    print("dino_pair:", c[0].shape, c[1].shape, "inliers", len(first), "weight", w)


def bunny18():
    ids = list(range(0, 36, 2))
    xyz, off, gt, init = [], [0], [], []
    rng = np.random.default_rng(0xB18)
    for k, i in enumerate(ids):
        c = np.loadtxt(f"{REF}/cloudXYZ_{i}.xyz")[:, :3]
        um = np.rint(c * 1e8).astype(np.int64)
        assert np.abs(um).max() < 2 ** 31 and np.array_equal(um.astype(np.float64) / 1e8, c), "int32 x 1e-8 m must be lossless"
        xyz.append(um.astype(np.int32)); off.append(off[-1] + len(c))
        P = np.loadtxt(f"{REF}/poses_{i}.txt")
        gt.append(P)
        Q = P.copy()
        if k > 0:   # addNoise (common.h:38-67): pose * SO3::exp(sigma w), translation += sigmat t
            Q[:3, :3] = P[:3, :3] @ synth._so3_exp(rng.normal(0.0, 1.0, 3) * 0.02)
            Q[:3, 3] = P[:3, 3] + rng.normal(0.0, 1.0, 3) * 0.01
        init.append(Q)
    np.savez_compressed(os.path.join(OUT, "bunny18.npz"), n_frames=len(ids), frame_ids=np.array(ids), offsets=np.array(off, np.int64),
                        xyz_e8=np.concatenate(xyz), poses_gt=np.stack(gt), poses_init=np.stack(init))
    print("bunny18:", off[-1], "points", os.path.getsize(os.path.join(OUT, "bunny18.npz")) / 1e6, "MB")


def lm_golden():
    sc = synth.make_scene(4, 3000, config_id=7)
    edges = synth.ring_edges(4, 2)
    idxs = [O.KdIndex(p, "kd") for p in sc["pts"]]
    corr, weights = [], []
    for s, d in edges:
        i, d2 = idxs[d].closest_points(sc["pts"][s], sc["poses_init"][s], sc["poses_init"][d])
        f, sec, dist, w, _ = O.filter_edge(i, d2, np.float32(0.05))
        corr.append((f, sec)); weights.append(w)
    out = {}
    for param in (0, 1, 2):
        for cost in (0, 1, 2):
            for robust in (0, 1):
                P, s, tr = O.optimize(sc["pts"], sc["nor"], sc["poses_init"], edges, corr, weights, param=param, cost=cost,
                                      robust=bool(robust), se3_autodiff=True, threads=1)
                k = f"p{param}_c{cost}_r{robust}"
                out[k + "_poses"] = P; out[k + "_trace"] = tr
                out[k + "_summary"] = np.array([s["termination"], s["num_iterations"], s["num_successful_steps"]], np.int64)
                out[k + "_cost"] = np.array([s["initial_cost"], s["final_cost"]])
                print(k, O.TERMINATION[s["termination"]], s["num_iterations"], s["initial_cost"], s["final_cost"])
    np.savez_compressed(os.path.join(OUT, "lm_golden.npz"), **out)


def sophus_vectors():
    # ext/sophus-ceres/test/core/test_se3.cpp:40-65: SE3(SO3::exp(w), t) ; :67-82 tangents (upsilon, omega)
    pi = np.pi
    el = [([0.2, 0.5, 0.0], [0, 0, 0]), ([0.2, 0.5, -1.0], [10, 0, 0]), ([0.0, 0.0, 0.0], [0, 100, 5]),
          ([0.0, 0.0, 0.00001], [0, 0, 0]), ([0.0, 0.0, 0.00001], [0, -0.00000001, 0.0000000001]),
          ([0.0, 0.0, 0.00001], [0.01, 0, 0]), ([pi, 0, 0], [4, -5, 0]),
          ([0.2, 0.5, 0.0], [0, 0, 0]), ([0.3, 0.5, 0.1], [2, 0, -7])]
    tg = [[0, 0, 0, 0, 0, 0], [1, 0, 0, 0, 0, 0], [0, 1, 0, 1, 0, 0], [0, -5, 10, 0, 0, 0], [-1, 1, 0, 0, 0, 1],
          [20, -1, 0, -1, 1, 0], [30, 5, -1, 20, -1, 0]]
    np.savez_compressed(os.path.join(OUT, "sophus_vectors.npz"), so3_omega=np.array([e[0] for e in el], float),
                        trans=np.array([e[1] for e in el], float), tangents=np.array(tg, float))


def ref_pins():
    import ctypes as C
    sys.path.insert(0, os.path.dirname(OUT))
    from test_oracle_functor_pin import _rand_pose
    assert O.ref_lib() is not None and O.ref_functors() is not None, "oracle/_ref was not built"
    out = {}
    sc = synth.make_scene(3, 20000, config_id=32)
    ref = O.KdIndex(sc["pts"][0], "ref")
    for name in ("poses_init", "poses_gt"):
        P = sc[name]
        idx, d2 = ref.closest_points(sc["pts"][1], P[1], P[0], threads=4)
        out[f"corr_{name}_idx"] = idx
        out[f"corr_{name}_d2_sha256"] = np.array(hashlib.sha256(d2.tobytes()).hexdigest())
    g = np.load(os.path.join(OUT, "bunny_pair.npz"))
    pts = g["pts0"]
    rf = O.KdIndex(pts, "ref")
    q = np.arange(0, len(pts), 53)
    res = [O.knn(rf, pts[i], 10) for i in q]
    out["knn_query"] = q
    out["knn_idx"] = np.stack([r[0] for r in res]); out["knn_d2"] = np.stack([r[1] for r in res])
    for param in (0, 1, 2):
        for plane in (0, 1):
            G = 6 if param == 0 else 7
            rng = np.random.default_rng(100 + 10 * param + plane)   # the loop of test_global_functors_match_reference_text
            ins, rs, js = [], [], []
            for it in range(32):
                c1 = _rand_pose(rng, param, unit=it % 3 != 0); c2 = _rand_pose(rng, param, unit=it % 3 != 0)
                if param == 0 and it % 50 == 0:
                    c1[:3] = rng.normal(0, 1e-9, 3)
                src = rng.normal(0, 0.3, 3); dst = rng.normal(0, 0.3, 3); nor = rng.normal(size=3); nor /= np.linalg.norm(nor)
                r, j = O.functor_eval(param, plane, c1, c2, src, dst, nor, "ref")
                ins.append(np.concatenate([c1, c2, src, dst, nor])); rs.append(r); js.append(j)
            k = f"gfun_p{param}_l{plane}"
            out[k + "_in"] = np.stack(ins); out[k + "_r"] = np.stack(rs); out[k + "_j"] = np.stack(js)
            rng = np.random.default_rng(200 + 10 * param + plane)   # the loop of test_pairwise_functors_are_the_global_ones_with_identity_dst
            ins, rs, js = [], [], []
            for it in range(16):
                c1 = _rand_pose(rng, param)
                src = rng.normal(0, 0.3, 3); dst = rng.normal(0, 0.3, 3); nor = rng.normal(size=3); nor /= np.linalg.norm(nor)
                r, j = O.functor_eval_pairwise_ref(param, plane, c1, src, dst, nor)
                ins.append(np.concatenate([c1, src, dst, nor])); rs.append(r); js.append(j)
            k = f"pfun_p{param}_l{plane}"
            out[k + "_in"] = np.stack(ins); out[k + "_r"] = np.stack(rs); out[k + "_j"] = np.stack(js)
    lib = O.ref_functors()
    P = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    rng = np.random.default_rng(7)   # the loop of test_quaternion_parameterisation_matches_reference_text
    xs, ds, pl, jac = [], [], [], []
    for it in range(40):
        x = rng.normal(size=4); x /= np.linalg.norm(x)
        d = rng.normal(0, 0.3, 3) if it % 10 else np.zeros(3)
        o = np.zeros(4); lib.ref_quat_plus(P(x), P(d), P(o))
        j = np.zeros(12); lib.ref_quat_jacobian(P(x), P(j))
        xs.append(x); ds.append(d); pl.append(o); jac.append(j)
    out.update(quat_x=np.stack(xs), quat_d=np.stack(ds), quat_plus=np.stack(pl), quat_jac=np.stack(jac))
    np.savez_compressed(os.path.join(OUT, "ref_pins.npz"), **out)
    print("ref_pins:", os.path.getsize(os.path.join(OUT, "ref_pins.npz")) / 1e3, "kB")


if __name__ == "__main__":
    only = sys.argv[1:]
    for fn in (bunny_pair, dino_pair, lm_golden, sophus_vectors, bunny18, ref_pins):
        if not only or fn.__name__ in only:
            fn()
