import os, sys, time, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
torch.cuda.init(); torch.zeros(1, device='cuda'); torch.cuda.synchronize()
import mv_lm_icp_b200 as mv
from mv_lm_icp_b200 import synth
import bench
sc = bench.load_scene(3, 20, 200000)
for rep in range(3):
    t0 = time.perf_counter(); eng = mv.Engine(); t1 = time.perf_counter()
    eng.set_frames(sc['pts'], sc['nor']); t2 = time.perf_counter()
    eng.set_graph(synth.ring_edges(20, 2)); t3 = time.perf_counter()
    eng.set_poses(sc['poses_init']); eng.sync(); t4 = time.perf_counter()
    print('rep', rep, 'create %.1f ms  set_frames %.1f ms  set_graph %.1f ms  set_poses %.1f ms' % ((t1-t0)*1e3, (t2-t1)*1e3, (t3-t2)*1e3, (t4-t3)*1e3))
    eng.close()
