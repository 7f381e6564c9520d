import numpy as np, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
from oracle import oracle as O
import mv_lm_icp_b200 as mv
from mv_lm_icp_b200.api import default_options
g = np.load(os.path.join(ROOT, 'tests', 'golden', 'bunny_pair.npz'))
pts = [g["pts0"], g["pts1"], g["pts0"][::2].copy()]; nor = [g["nor0"], g["nor1"], g["nor0"][::2].copy()]
bump = np.eye(4); bump[:3, :3] = np.array([[1, -0.004, 0.003], [0.004, 1, -0.002], [-0.003, 0.002, 1]]); bump[:3, 3] = [0.002, -0.001, 0.0015]
poses0 = np.stack([g["pose0"], g["pose1"], bump @ g["pose0"]])
edges = [(1, 0), (1, 2), (2, 1), (2, 0)]
for param in (2, 1):
  for cost in (0, 1):
    eng = mv.Engine(); eng.set_frames(pts, nor); eng.set_graph(edges)
    poses = poses0.copy()
    for rnd in range(3):
      eng.set_poses(poses); eng.correspond(0.05)
      corr=[]; w=[]
      for e in range(len(edges)):
          f,s,d,ww = eng.get_edge(e); corr.append((f,s)); w.append(ww)
      s = eng.optimize(param, cost, True); P = eng.get_poses()
      Pr, sr, tr = O.optimize(pts, nor, poses, edges, corr, w, param=param, cost=cost, robust=True, se3_autodiff=True, threads=8)
      print('param', param, 'cost', cost, 'round', rnd, 'iters', s['num_iterations'], sr['num_iterations'], 'term', s['termination'], sr['termination'],
            'cost0 %.10e %.10e' % (s['initial_cost'], sr['initial_cost']), 'costF %.10e %.10e' % (s['final_cost'], sr['final_cost']), 'pose %.2e' % np.abs(P-Pr).max())
      print('   trace', [(int(r[0]), int(r[1]), int(r[2]), '%.6e' % r[4], '%.1e' % r[7]) for r in tr[:8]])
      poses = Pr
    eng.close()
