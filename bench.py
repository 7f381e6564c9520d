#!/usr/bin/env python
"""bench.py -- outer ICP iterations / second (correspondence + LM) on BASELINE.json's config.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5|real]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One "step" = one pass of the loop body main_multiview.cpp:150-169 minus rendering: correspondences of every frame
(Frame::computeClosestPointsToNeighbours) + one full LM solve (ceresOptimizer*).  The K timed steps are the first K
rounds of the real ICP trajectory from the seeded noisy poses (the reference hard-codes 20); the W warm-up steps run
the same rounds beforehand and the poses are then reset, so warm-up does not change the timed work.
Default workload = BASELINE.json configs[2] (the config the metric is quoted on): 20 views x 200k pts, point-to-plane,
Sophus SE(3), robust, cutoff 0.05, knn 2, synthetic bunny-shaped scans (mv_lm_icp_b200/synth.py).  `--config real` is
the reference's default invocation (main_multiview.cpp:33-36,63): the 18 real Bunny_RealData frames 0,2,..,34 with
their (non-rigid) sample poses + seeded noise, recomputed normals, pose-graph knn 2 (tests/golden/bunny18.npz).

Both arms print, per round, the inlier count and the LM iteration count, and a sha256 of the final poses: the
reference arm leaves them in /tmp for the GPU arm that follows it on the same box, which reports whether both arms did
the same work (BASELINE.md section 3) -- the driver computes the ratio, this file only says whether it is meaningful.
"""
import argparse
import hashlib
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {   # BASELINE.json configs[] (index = config id); knn = 2 everywhere (main_multiview.cpp:41)
    "2": dict(views=10, points=100_000, param="aa", cost="p2plane"),
    "3": dict(views=20, points=200_000, param="se3", cost="p2plane"),
    "4": dict(views=40, points=500_000, param="quat", cost="mixed"),
    "5": dict(views=64, points=1_000_000, param="se3", cost="p2plane"),
    "0": dict(views=6, points=20_000, param="se3", cost="p2plane"),   # tiny, for dry runs
    "real": dict(views=18, points=None, param="se3", cost="p2plane"),
}
PARAM = {"aa": 0, "quat": 1, "se3": 2}
COST = {"p2p": 0, "p2plane": 1, "mixed": 2}
CUTOFF = 0.05


def workload_name(cid, cfg):
    if cid == "real":
        return ("multiview point-to-plane, 18 real Bunny_RealData frames (0,2,..,34: 224673 pts), se3 param, robust, knn 2, cutoff 0.05, "
                "recomputed normals (the reference's default invocation, main_multiview.cpp:33-51)")
    tag = {"2": " (BASELINE configs[1])", "3": " (BASELINE configs[2])", "4": " (BASELINE configs[3])", "5": " (BASELINE configs[4])"}.get(cid, "")
    cost = {"p2plane": "point-to-plane", "p2p": "point-to-point", "mixed": "point-to-point+plane mixed"}[cfg["cost"]]
    return f"multiview {cost}, {cfg['views']} views x {cfg['points']} pts, {cfg['param']} param, robust, knn 2, cutoff 0.05{tag}"


# ======================================================================================================
# host resources
# ======================================================================================================
def cpu_threads():
    """Threads for the CPU arm: the CPUs this process may run on (affinity), capped by the cgroup CPU quota and by the
    physical core count (hyper-thread siblings slow the static-schedule loops down).  OMP_NUM_THREADS is ignored on
    purpose: torchrun exports OMP_NUM_THREADS=1, which would silently turn the all-core figure into a 1-thread one."""
    n = len(os.sched_getaffinity(0))
    try:   # cgroup v2
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(math.floor(float(q) / float(p)))))
    except Exception:
        try:   # cgroup v1
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:
            pass
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
        if phys:
            n = min(n, phys)
    except Exception:
        pass
    return max(1, n)


def _gen_view(a):
    from mv_lm_icp_b200 import synth
    v, views, points, cid = a
    try:   # one BLAS thread per worker: the pool already fills the CPUs this process may use
        from threadpoolctl import threadpool_limits
        with threadpool_limits(limits=1):
            p, n, P = synth.make_view(v, views, points, 0xB200 + 1000 * cid + v)
    except ImportError:
        p, n, P = synth.make_view(v, views, points, 0xB200 + 1000 * cid + v)
    return v, p, n


def load_scene(cid, cfg, rank=0, world=1, barrier=None):
    """Seeded synthetic scene (or the real-frame fixture), cached under /tmp.  With several ranks every rank generates
    its share of the views (a process pool each) and all ranks then read the cached files."""
    if cid == "real":
        z = np.load(os.path.join(ROOT, "tests", "golden", "bunny18.npz"))
        M = int(z["n_frames"])
        off = z["offsets"]; xyz = z["xyz_e8"].astype(np.float64) / 1e8     # <= 8-decimal text -> exact doubles (correctly rounded division)
        pts = [np.ascontiguousarray(xyz[off[i]:off[i + 1]]) for i in range(M)]
        return {"pts": pts, "nor": [None] * M, "poses_gt": z["poses_gt"], "poses_init": z["poses_init"], "real": True}
    from mv_lm_icp_b200 import synth
    views, points = cfg["views"], cfg["points"]
    icid = int(cid)
    base = f"/tmp/mvicp_scene_c{cid}_{views}x{points}"
    mine = [v for v in range(views) if v % world == rank and not os.path.exists(f"{base}_v{v}.npz")]
    if mine:
        workers = max(1, min(len(mine), cpu_threads() // max(1, world), 16 if points >= 400_000 else 32))
        if workers > 1:
            import multiprocessing as mp
            with mp.get_context("fork").Pool(workers) as pool:
                res = pool.map(_gen_view, [(v, views, points, icid) for v in mine])
        else:
            res = [_gen_view((v, views, points, icid)) for v in mine]
        for v, p, n in res:
            tmp = f"{base}_v{v}.{os.getpid()}.tmp.npz"
            np.savez(tmp, p=p.astype(np.float32), n=n.astype(np.float32))   # every value is fp32-exact by construction
            os.replace(tmp, f"{base}_v{v}.npz")
    if barrier is not None:
        barrier()
    pts, nor = [], []
    for v in range(views):
        z = np.load(f"{base}_v{v}.npz")
        pts.append(z["p"].astype(np.float64)); nor.append(z["n"].astype(np.float64))
    gt, init = synth.scene_poses(views, icid)
    return {"pts": pts, "nor": nor, "poses_gt": gt, "poses_init": init, "real": False}


def scene_graph(sc, cfg):
    """Edge list as Frame::computePoseNeighboursKnn yields it from the initial poses (frame.cpp:67-89)."""
    from mv_lm_icp_b200 import synth
    if sc.get("real"):
        P = sc["poses_init"]
        edges = []
        for i in range(len(P)):
            d = [(np.float32(np.linalg.norm(P[i][:3, 3] - P[j][:3, 3])), j) for j in range(len(P)) if j != i]
            d.sort(key=lambda x: x[0])   # stable: ties keep the lower index
            edges += [(i, d[0][1]), (i, d[1][1])]
        return edges
    return synth.ring_edges(cfg["views"], 2)


def pose_sha(P):
    return hashlib.sha256(np.ascontiguousarray(np.asarray(P, dtype=np.float64)).tobytes()).hexdigest()


LM_SUMMARY_FIELDS = ("termination", "num_iterations", "num_successful_steps", "num_evaluations", "num_linear_solves",
                     "initial_cost", "final_cost")
NN_SAMPLE_ROWS = 1_500_000   # 4 float64 columns: 48 MB, which keeps the whole dump under 64 MB
NN_SAMPLE_SEED = 0xD0


def dump_outputs(out_dir, eng, sc, edges, poses, summary, world):
    """What the last timed step handed its caller, as .npy files in out_dir, so that two builds run with the same arguments can be
    compared output for output: poses.npy (float64 [M, 4, 4]) and lm_summary.npy (float64, LM_SUMMARY_FIELDS in that order); with
    one GPU, per edge edge_inliers.npy / edge_weights.npy (float64 / float32 [E]) and, for a fixed seeded sample of every free
    frame's queries, nn_edge / nn_query / nn_idx / nn_d2.npy (float64 [rows]): the edge, the query point, its nearest neighbour in
    the destination frame and their squared distance (every list in full would exceed 64 MB at configs 3-5)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "poses.npy"), np.asarray(poses, np.float64))
    np.save(os.path.join(out_dir, "lm_summary.npy"), np.array([summary[k] for k in LM_SUMMARY_FIELDS], np.float64))
    if world > 1:     # a rank holds the correspondences of its own edges only
        return
    cw = [eng.get_edge(e, arrays=False) for e in range(len(edges))]
    np.save(os.path.join(out_dir, "edge_inliers.npy"), np.array([c for c, _ in cw], np.float64))
    np.save(os.path.join(out_dir, "edge_weights.npy"), np.array([w for _, w in cw], np.float32))
    act = [e for e, (s, _) in enumerate(edges) if s != 0]
    rng = np.random.default_rng(NN_SAMPLE_SEED)
    cols = {"nn_edge": [], "nn_query": [], "nn_idx": [], "nn_d2": []}
    for e in act:
        n = len(sc["pts"][edges[e][0]])
        q = np.sort(rng.choice(n, min(n, NN_SAMPLE_ROWS // len(act)), replace=False))
        idx, d2 = eng.get_nn(e)
        cols["nn_edge"].append(np.full(len(q), e, np.float64)); cols["nn_query"].append(q.astype(np.float64))
        cols["nn_idx"].append(idx[q].astype(np.float64)); cols["nn_d2"].append(d2[q])
    for k, v in cols.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.concatenate(v) if v else np.zeros(0))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (profiling guide's clocks line)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.idx = gpu_index; self.samples = []; self.stop_flag = False; self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append(line.strip())
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def measured_traffic(kernel):
    """DRAM bytes per launch of a kernel from the committed `ncu --set full` capture (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p)).get(kernel)
    except Exception:
        return None


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ======================================================================================================
# CPU arm: the reference path on the host cores (nanoflann verbatim from oracle/_ref when built, oracle LM port)
# ======================================================================================================
class CpuArm:
    """The whole problem (every edge with a free src frame), round by round, as main_multiview.cpp:150-169 runs it."""

    def __init__(self, sc, cfg, edges):
        from oracle import oracle as O
        self.O = O; self.sc = sc; self.cfg = cfg; self.edges = edges
        self.kind = "ref" if O.ref_lib() is not None else "kd"
        self.act = [(e, s, d) for e, (s, d) in enumerate(edges) if s != 0]
        t0 = time.perf_counter()
        self.idx = {d: O.KdIndex(sc["pts"][d], self.kind) for d in sorted(set(d for _, _, d in self.act))}   # one-time build: excluded, as the reference's lazily built index is amortised
        self.build_s = time.perf_counter() - t0
        self.nor = sc["nor"]

    def ensure_normals(self, threads):
        if self.nor[0] is None:   # Frame::recomputeNormals (main_multiview.cpp:68), not part of the metric
            self.nor = [self.O.recompute_normals(p, 10, threads=threads) for p in self.sc["pts"]]

    def round(self, poses, threads):
        """One outer round from `poses`: returns (new poses, corr seconds, LM seconds, inliers, LM iterations)."""
        O = self.O
        t0 = time.perf_counter()
        corr = [(np.zeros(0, np.int32), np.zeros(0, np.int32))] * len(self.edges); w = [0.0] * len(self.edges)
        inl = 0
        for e, s, d in self.act:
            i, d2 = self.idx[d].closest_points(self.sc["pts"][s], poses[s], poses[d], threads=threads)
            f, sec, dist, ww, _ = O.filter_edge(i, d2, np.float32(CUTOFF))
            corr[e] = (f, sec); w[e] = ww; inl += len(f)
        t1 = time.perf_counter()
        new, summ, _ = O.optimize(self.sc["pts"], self.nor, poses, self.edges, corr, w, param=PARAM[self.cfg["param"]],
                                  cost=COST[self.cfg["cost"]], robust=True, se3_autodiff=True, threads=threads)
        t2 = time.perf_counter()
        return new, t1 - t0, t2 - t1, inl, summ["num_iterations"]

    def run(self, n_rounds, threads, poses=None):
        poses = self.sc["poses_init"].copy() if poses is None else poses
        rec = []
        for _ in range(n_rounds):
            poses, a, b, inl, it = self.round(poses, threads)
            rec.append(dict(corr_s=a, lm_s=b, inliers=int(inl), lm_iters=int(it)))
        return poses, rec

    def nn_name(self):
        return "reference nanoflann.hpp (oracle/_ref)" if self.kind == "ref" else "oracle KD-tree port"


def trace_path(cid):
    return f"/tmp/mvicp_refarm_c{cid}.json"


def run_reference(args, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = cpu_threads()
    sc = load_scene(args.config, cfg)
    edges = scene_graph(sc, cfg)
    arm = CpuArm(sc, cfg, edges)
    arm.ensure_normals(threads)
    if args.warmup > 0:
        arm.run(1, threads)      # page in code and data; CPU timings do not drift after that
    poses, rec = arm.run(args.steps, threads)                 # all edges, all K rounds, every core this process may use
    # the reference itself is single-threaded (no OpenMP, Ceres num_threads = 1): the faithful figure, on the first rounds of
    # the same problem (a round costs ~45 s on one thread at config 3; --single-rounds K for all of them)
    n1 = min(args.steps, args.single_rounds)
    poses1, rec1 = arm.run(n1, 1) if n1 > 0 else (None, [])
    per_round = float(np.mean([r["corr_s"] + r["lm_s"] for r in rec]))
    val = 1.0 / per_round
    E_act = len(arm.act); Q = sum(len(sc["pts"][s]) for _, s, _ in arm.act)
    sample = (f"rounds 0..{args.steps - 1} of the whole problem ({E_act} directed edges with a free src frame, {Q} queries per round; "
              f"{'one untimed warm-up round' if args.warmup > 0 else 'no warm-up'}); NN = {arm.nn_name()}, LM = oracle port of the Ceres path "
              f"(Jet autodiff, dense Cholesky; Ceres not installable), {threads} OpenMP threads (affinity/cgroup/physical-core cap, "
              f"OMP_NUM_THREADS ignored); index build ({arm.build_s:.2f} s) excluded")
    trace = {"inliers_per_round": [r["inliers"] for r in rec], "lm_iterations_per_round": [r["lm_iters"] for r in rec],
             "pose_sha": pose_sha(poses), "final_poses": np.asarray(poses).tolist(), "steps": args.steps, "threads": threads}
    try:
        json.dump(trace, open(trace_path(args.config), "w"))
    except Exception:
        pass
    cb = {"value": val, "unit": "iter/s", "cores": threads, "kind": "reference" if arm.kind == "ref" else "port", "sample": sample,
          "corr_s_per_round": float(np.mean([r["corr_s"] for r in rec])), "lm_s_per_round": float(np.mean([r["lm_s"] for r in rec]))}
    if rec1:
        pr1 = float(np.mean([r["corr_s"] + r["lm_s"] for r in rec1]))
        pra = float(np.mean([r["corr_s"] + r["lm_s"] for r in rec[:n1]]))
        cb["single_thread"] = {"value": 1.0 / pr1, "unit": "iter/s", "cores": 1,
                               "sample": f"rounds 0..{n1 - 1} of the same problem on one thread", "all_core_value_same_rounds": 1.0 / pra,
                               "corr_s_per_round": float(np.mean([r["corr_s"] for r in rec1])), "lm_s_per_round": float(np.mean([r["lm_s"] for r in rec1])),
                               "lm_iterations_per_round": [r["lm_iters"] for r in rec1], "inliers_per_round": [r["inliers"] for r in rec1],
                               "same_counts_as_all_core": [r["inliers"] for r in rec1] == [r["inliers"] for r in rec[:n1]] and
                                                          [r["lm_iters"] for r in rec1] == [r["lm_iters"] for r in rec[:n1]]}
    out = {"impl": "reference", "metric": "ICP iterations/sec (corr+LM)", "value": val, "unit": "iter/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_round * 1e3, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f64", "data": "real scans (tests/golden/bunny18.npz)" if sc.get("real") else "synthetic",
           "config": {"workload": workload_name(args.config, cfg)},
           "cpu_baseline": cb, "inliers_per_round": trace["inliers_per_round"], "lm_iterations_per_round": trace["lm_iterations_per_round"],
           "pose_sha": trace["pose_sha"],
           "e2e": {"value": val, "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(out), flush=True)


# ======================================================================================================
# GPU arm
# ======================================================================================================
def _file_barrier(cid, cfg, timeout_s=3600):
    """Ranks generate disjoint shares of the scene BEFORE torch / NCCL / CUDA are initialised (the generator forks a process
    pool); they meet again when every view's file exists (files appear by atomic rename)."""
    def wait():
        base = f"/tmp/mvicp_scene_c{cid}_{cfg['views']}x{cfg['points']}"
        t0 = time.time()
        while not all(os.path.exists(f"{base}_v{v}.npz") for v in range(cfg["views"])):
            if time.time() - t0 > timeout_s:
                raise RuntimeError("scene generation: another rank never delivered its views")
            time.sleep(0.2)
    return wait


def run_ours(args, cfg):
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    sc = load_scene(args.config, cfg, rank, world, _file_barrier(args.config, cfg) if (world > 1 and args.config != "real") else None)
    import torch
    import mv_lm_icp_b200 as mv
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    dev = local if world > 1 else 0
    torch.cuda.set_device(dev)

    M = len(sc["pts"]); n_pts = [len(p) for p in sc["pts"]]
    edges = scene_graph(sc, cfg)
    param, cost = PARAM[cfg["param"]], COST[cfg["cost"]]

    def make_engine(with_comm):
        t0 = time.perf_counter()
        eng = mv.Engine(device=dev, flags=args.flags)
        eng.set_frames(sc["pts"], None if sc["nor"][0] is None else sc["nor"])
        nms = None
        if sc["nor"][0] is None:
            _, nms = eng.recompute_normals(10, fetch=False)      # Frame::recomputeNormals (main_multiview.cpp:68)
        eng.set_poses(sc["poses_init"])
        eng.set_graph(edges)
        comm_s = 0.0
        if with_comm and world > 1:
            eng.sync(); t1 = time.perf_counter()
            idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == 0:
                idt.copy_(torch.frombuffer(bytearray(mv.nccl_unique_id()), dtype=torch.uint8))
            dist.broadcast(idt, 0)
            eng.comm_init(bytes(idt.cpu().numpy().tobytes()), rank, world)
            eng.sync(); comm_s = time.perf_counter() - t1
        eng.sync()
        make_engine.comm_s = comm_s      # NCCL communicator + peer-memory mapping: once per process group, not per scene
        return eng, time.perf_counter() - t0 - comm_s, nms

    eng, setup_s, normals_ms = make_engine(True)
    comm_init_s = make_engine.comm_s
    # Frame::recomputeNormals (default-on in the reference, before round 0; not part of the metric): timed once, on a
    # scratch engine so that the synthetic benchmark itself keeps the uploaded fp32-exact normals
    if rank == 0 and world == 1 and normals_ms is None and not args.no_normals:
        e2 = mv.Engine(device=dev); e2.set_frames(sc["pts"], sc["nor"])
        e2.recompute_normals(10, fetch=False); _, normals_ms = e2.recompute_normals(10, fetch=False)
        e2.close()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(); eng.sync()

    def run_rounds(en, k, mode, stream, instrument=True):
        """k rounds from the initial poses.  mode: 'dev' (poses stay on the device), 'e2e' (poses cross the C ABI as host buffers every
        step), 'mat' (e2e + every correspondence list materialised on the host, as frame.cpp:158 does).
        instrument=True: per-round device ms (events on the engine's stream), a sync and the engine's stats after every round -- the
        breakdown passes.  instrument=False: nothing but the calls a user makes -- the TIMED passes (per = bytes per round only)."""
        en.set_graph(edges)             # forget the previous trajectory's matches: round 0 is a cold, unseeded search
        en.set_poses(sc["poses_init"])
        per = []
        poses = sc["poses_init"]
        traj = []
        if not instrument:
            for r in range(k):
                if mode != "dev":
                    en.set_poses(poses)        # host buffer -> device, through the C ABI
                if mode == "mat":
                    en.correspond(CUTOFF)
                    nb = en.pull_all_edges()
                    s = en.optimize(param, cost, True)
                else:
                    nb = 0
                    s = en.icp_round(CUTOFF, param, cost, True)
                if mode != "dev":
                    poses = en.get_poses()     # device -> host
                per.append(dict(d2h=nb, summary=s))
            en.sync()
            return per, traj
        for r in range(k):
            ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            ev0.record(stream)
            if mode != "dev":
                en.set_poses(poses)        # host buffer -> device, through the C ABI
            if mode == "mat":
                en.correspond(CUTOFF)
                nb = en.pull_all_edges()
                s = en.optimize(param, cost, True)
            else:
                nb = 0
                s = en.icp_round(CUTOFF, param, cost, True)
            if mode != "dev":
                poses = en.get_poses()     # device -> host
            ev1.record(stream)
            en.sync()
            wall = time.perf_counter() - t0
            st = en.stats()
            per.append(dict(ms=ev0.elapsed_time(ev1), wall_ms=wall * 1e3, lm_iters=s["num_iterations"], evals=s["num_evaluations"],
                            knn_ms=st["knn_ms"], select_ms=st["select_ms"], lm_eval_ms=st["lm_eval_ms"], lm_other_ms=st["lm_other_ms"],
                            corr=st["correspondences"], queries=st["queries"], d2h=nb))
            if args.check_cpu and mode == "dev":
                traj.append(en.get_poses())
        return per, traj

    stream = torch.cuda.ExternalStream(eng.stream(), device=dev)
    # warm-up (untimed), then EXACTLY K timed steps between barriers
    run_rounds(eng, max(3, args.warmup), "dev", stream)
    sampler = ClockSampler(dev); sampler.start(); time.sleep(0.3)
    barrier()
    st0 = eng.stats(); l0 = st0["kernel_launches"]
    t0 = time.perf_counter()
    timed, _ = run_rounds(eng, args.steps, "dev", stream, instrument=False)     # the timed K steps: nothing but the K calls
    barrier()
    wall_total = time.perf_counter() - t0
    st1 = eng.stats(); l1 = st1["kernel_launches"]
    final_poses = eng.get_poses()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, sc, edges, final_poses, timed[-1]["summary"], world)
    # e2e: same K rounds, poses cross the C ABI as host buffers every step
    barrier()
    t0 = time.perf_counter()
    run_rounds(eng, args.steps, "e2e", stream, instrument=False)
    barrier()
    wall_e2e = time.perf_counter() - t0
    wall_mat = None; per_mat = None
    if world == 1 and not args.no_mat:
        barrier()
        t0 = time.perf_counter()
        per_mat, _ = run_rounds(eng, args.steps, "mat", stream, instrument=False)
        barrier()
        wall_mat = time.perf_counter() - t0
    # the same K rounds once more, instrumented (events, a sync and the engine's stats after every round): the per-round / per-kernel
    # breakdown and the inlier / LM-iteration counts.  Same work, same poses -- checked.
    barrier()
    per, _ = run_rounds(eng, args.steps, "dev", stream)
    if pose_sha(eng.get_poses()) != pose_sha(final_poses):
        raise SystemExit("bench.py: the instrumented pass ended on different poses than the timed pass")
    clocks = sampler.finish()       # sampled over the timed passes and the instrumented repeat (same kernels, same load)
    traj = None
    if args.check_cpu and world == 1:
        _, traj = run_rounds(eng, args.steps, "dev", stream)

    dev_ms = sum(p["ms"] for p in per)
    tot = torch.tensor([dev_ms, wall_total * 1e3, wall_e2e * 1e3], dtype=torch.float64, device="cuda")
    inl = torch.tensor([p["corr"] for p in per], dtype=torch.int64, device="cuda")   # inliers of this rank's edges, per round
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        dist.all_reduce(inl, op=dist.ReduceOp.SUM)
    dev_ms, wall_ms, e2e_ms = [float(x) for x in tot.cpu()]
    inliers = [int(x) for x in inl.cpu()]
    mine = {k: round(sum(p[k] for p in per) / args.steps, 4) for k in ("knn_ms", "select_ms", "lm_eval_ms", "lm_other_ms")}
    mine["queries"] = int(per[0]["queries"])
    per_rank = [mine]
    sha = pose_sha(final_poses)
    shas = [sha]
    if world > 1:   # lm_other of a rank includes its wait for the slowest rank's matrices: the imbalance shows here
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
        shas = [None] * world
        dist.all_gather_object(shas, sha)
    # multi-GPU correctness, visible to whoever reads the line: rank 0 replays the same K rounds alone on its GPU (no
    # communicator) and the poses of the sharded run must be the same bytes (DESIGN section 5: bit-identical for any N)
    sha_1gpu = None
    if world > 1 and rank == 0 and not args.no_replay:
        solo, _, _ = make_engine(False)
        run_rounds(solo, args.steps, "dev", torch.cuda.ExternalStream(solo.stream(), device=dev))
        sha_1gpu = pose_sha(solo.get_poses())
        solo.close()
    if world > 1:
        dist.barrier()    # the other ranks wait for rank 0's replay before anybody tears its communicator down
    if rank == 0:
        peak, peak_src = hbm_peak()
        K = args.steps
        # the step is host-driven (one sync per LM iteration), so the honest whole-step time is the wall clock between the barriers
        ms_per_step = wall_ms / K
        knn_ms = float(np.mean([p["knn_ms"] for p in per]))
        q_local = per[0]["queries"]
        knn_bytes = 44.0 * q_local
        evals = sum(p["evals"] for p in per); lm_eval_ms = sum(p["lm_eval_ms"] for p in per)
        corr_mean = float(np.mean([p["corr"] for p in per]))
        lm_bytes = 52.0 * corr_mean if cost != 0 else 36.0 * corr_mean
        knn_gbs = knn_bytes / (knn_ms * 1e-3) / 1e9
        lm_gbs = lm_bytes / ((lm_eval_ms / max(1, evals)) * 1e-3) / 1e9
        share = {"knn": sum(p["knn_ms"] for p in per) / dev_ms, "select": sum(p["select_ms"] for p in per) / dev_ms,
                 "lm_eval": lm_eval_ms / dev_ms, "lm_other": sum(p["lm_other_ms"] for p in per) / dev_ms}
        dominant = "knn" if share["knn"] >= share["lm_eval"] else "lm_eval"
        knn_name = "knn_kernel"      # the NN step of a round: knn_far_kernel (rounds 0-1), knn_kernel, or knn_cert_kernel + knn_todo_kernel (certified rounds)
        roof_knn = {"kernel": knn_name, "bound": "hbm", "achieved": knn_gbs, "peak": peak, "unit": "GB/s", "frac": knn_gbs / peak,
                    "traffic": measured_traffic(knn_name) if world == 1 else None, "algorithmic_bytes_per_launch": knn_bytes,
                    "avg_launch_ms": knn_ms, "peak_source": peak_src,
                    "frac_per_round": [round(44.0 * p["queries"] / (p["knn_ms"] * 1e-3) / 1e9 / peak, 4) for p in per]}
        roof_lm = {"kernel": "lm_eval_kernel", "bound": "hbm", "achieved": lm_gbs, "peak": peak, "unit": "GB/s", "frac": lm_gbs / peak,
                   "traffic": measured_traffic("lm_eval_kernel") if world == 1 else None, "algorithmic_bytes_per_launch": lm_bytes,
                   "avg_launch_ms": lm_eval_ms / max(1, evals), "peak_source": peak_src}
        pose_bytes = M * 16 * 8
        n_q = sum(n_pts[s] for s, _ in edges)
        out = {"metric": "ICP iterations/sec (corr+LM)", "value": 1e3 / ms_per_step, "unit": "iter/s", "n_gpus": world, "steps": K,
               "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f64", "data": "real scans (tests/golden/bunny18.npz)" if sc.get("real") else "synthetic",
               "config": {"workload": workload_name(args.config, cfg),
                          "l2": "no flush: resident working set (clouds + trees + match arrays) = %.0f MB > 126 MB L2" %
                                ((sum(n_pts) * 48 + n_q * 12) / 1e6),
                          "parallelism": f"edges (frame -> neighbour query sets) sharded over {world} GPU(s), one process per GPU",
                          "timing_passes": "value / e2e: K calls between barriers, nothing else in the loop; per-round and per-kernel figures: the same K rounds repeated with events + sync + stats per round (same final poses, checked)",
                          "timing": "wall clock between barriers (host-driven LM loop); device-event sum = %.3f ms/step" % (dev_ms / K),
                          "setup_ms_excluded": setup_s * 1e3, "comm_init_ms_excluded": comm_init_s * 1e3,
                          "normals_ms_excluded": normals_ms,
                          "per_round_ms": [round(p["ms"], 3) for p in per],
                          "per_round_knn_ms": [round(p["knn_ms"], 3) for p in per],
                          "per_rank_ms_per_step": per_rank,
                          "engine_flags": args.flags,
                          "storage": "fp64 records (real scans are not fp32-representable)" if sc.get("real") else "fp32 records (lossless), fp64 arithmetic"},
               "inliers_per_round": inliers, "lm_iterations_per_round": [p["lm_iters"] for p in per], "pose_sha": sha,
               "e2e": {"value": 1e3 / (e2e_ms / K), "unit": "iter/s", "h2d_bytes_per_step": pose_bytes, "d2h_bytes_per_step": pose_bytes,
                       "note": "per step: poses host->device, correspond+optimize, poses device->host through the C ABI; clouds uploaded once "
                               "(setup_ms_excluded), as the reference keeps its clouds and KD-trees across rounds",
                       "incl_setup_value": 1e3 / ((e2e_ms + setup_s * 1e3) / K)},
               "gpu_launches": int(l1 - l0), "clocks": clocks,
               "select_guess": {"rounds": int(st1["select_guess_rounds"] - st0["select_guess_rounds"]),
                                "edge_misses": int(st1["select_guess_misses"] - st0["select_guess_misses"])},
               "certified_matches": {"rounds": int(st1["cert_rounds"] - st0["cert_rounds"]),
                                     "kept_queries": int(st1["cert_reused"] - st0["cert_reused"]),
                                     "kept_fraction_in_those_rounds": round((st1["cert_reused"] - st0["cert_reused"]) / max(1, (st1["cert_rounds"] - st0["cert_rounds"]) * st1["queries"]), 4)},
               "roofline": roof_knn if dominant == "knn" else roof_lm, "roofline_knn": roof_knn, "roofline_lm": roof_lm,
               "time_share": share}
        if wall_mat is not None:
            out["e2e"]["materialized"] = {"value": 1e3 / (wall_mat * 1e3 / K), "unit": "iter/s", "d2h_bytes_per_step": int(np.mean([p["d2h"] for p in per_mat])) + pose_bytes,
                                          "note": "as e2e, plus every edge's (first, second, dist) list and weight copied to host vectors each round "
                                                  "(what Frame::computeClosestPointsToNeighbours leaves in OutgoingEdge::correspondances, frame.cpp:158)"}
        if world > 1:
            out["pose_sha_per_rank_equal"] = bool(all(s == sha for s in shas))
            out["pose_sha_1gpu_replay"] = sha_1gpu
            out["bit_identical_to_1gpu"] = (sha_1gpu == sha) if sha_1gpu is not None else None
        # the reference arm ran before this one on the same box (driver order): did both arms do the same work?
        try:
            ref = json.load(open(trace_path(args.config)))
            k2 = min(K, ref["steps"])
            pd = float(np.max(np.abs(np.asarray(ref["final_poses"]) - final_poses))) if ref["steps"] == K else None
            out["same_work_as_reference_arm"] = {
                "inliers_equal": ref["inliers_per_round"][:k2] == inliers[:k2],
                "lm_iterations_equal": ref["lm_iterations_per_round"][:k2] == out["lm_iterations_per_round"][:k2],
                "reference_inliers_per_round": ref["inliers_per_round"][:k2], "reference_lm_iterations_per_round": ref["lm_iterations_per_round"][:k2],
                "final_pose_max_abs_diff": pd, "rounds_compared": k2}
        except Exception:
            out["same_work_as_reference_arm"] = None
        if world == 1 and not args.no_cpu:
            th = cpu_threads()
            arm = CpuArm(sc, cfg, edges)
            arm.ensure_normals(th)
            n_s = 2 if n_q <= 10_000_000 else 1
            _, rec = arm.run(n_s, th)
            per_round = float(np.mean([r["corr_s"] + r["lm_s"] for r in rec]))
            out["cpu_baseline"] = {"value": 1.0 / per_round, "unit": "iter/s", "cores": th, "kind": "reference" if arm.kind == "ref" else "port",
                                   "sample": f"rounds 0..{n_s - 1} of the whole problem ({len(arm.act)} edges, {n_q} queries per round); NN = {arm.nn_name()}, "
                                             f"LM = oracle port (Ceres not installable), {th} threads; `--impl reference` times all {K} rounds and one thread too",
                                   "inliers_per_round": [r["inliers"] for r in rec], "lm_iterations_per_round": [r["lm_iters"] for r in rec],
                                   "same_work": [r["inliers"] for r in rec] == inliers[:n_s] and [r["lm_iters"] for r in rec] == out["lm_iterations_per_round"][:n_s]}
        if traj is not None:   # --check-cpu: every round replayed on the CPU from the GPU's own poses (same inputs => same counts)
            arm = CpuArm(sc, cfg, edges); th = cpu_threads(); arm.ensure_normals(th)
            chk = []
            poses = sc["poses_init"]
            for r in range(K):
                newp, _, _, inl_c, it_c = arm.round(poses, th)
                chk.append(dict(round=r, inliers_cpu=inl_c, inliers_gpu=inliers[r], lm_iters_cpu=it_c, lm_iters_gpu=per[r]["lm_iters"],
                                pose_max_abs_diff=float(np.max(np.abs(newp - traj[r])))))
                poses = traj[r]
            out["cpu_check_per_round"] = chk
        print(json.dumps(out), flush=True)
        if world > 1 and (not all(s == sha for s in shas) or (sha_1gpu is not None and sha_1gpu != sha)):
            raise SystemExit("bench.py: the sharded run's poses differ from the 1-GPU replay / between ranks")
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="3", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-mat", action="store_true", help="skip the e2e leg that materialises the correspondence lists on the host")
    ap.add_argument("--no-normals", action="store_true", help="skip timing the normal estimation")
    ap.add_argument("--no-replay", action="store_true", help="multi-GPU: skip rank 0's 1-GPU replay (bit-identity check)")
    ap.add_argument("--single-rounds", type=int, default=2, help="reference arm: rounds of the single-thread leg (0: skip)")
    ap.add_argument("--check-cpu", action="store_true", help="replay every round on the CPU from the GPU's poses and compare counts / poses")
    ap.add_argument("--flags", type=int, default=0, help="MVICP_FLAG_* bits for the engine (A/B measurements)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed to DIR/<name>.npy "
                                                           "(poses, LM summary, per-edge counts / weights, a seeded sample of the NN answers)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, cfg)
    else:
        run_ours(args, cfg)


if __name__ == "__main__":
    main()
