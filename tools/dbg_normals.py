import numpy as np, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
from oracle import oracle as O
import mv_lm_icp_b200 as mv
g = np.load(os.path.join(ROOT, 'tests', 'golden', 'bunny_pair.npz'))
pts = [g["pts0"], g["pts1"]]
eng = mv.Engine(); eng.set_frames(pts, [g["nor0"], g["nor1"]])
nor, ms = eng.recompute_normals(10)
nn = eng.knn_self(1, 10)
ref, rnn = O.recompute_normals(pts[1], 10, threads=8, want_nn=True)
bad = np.where(np.any(nn != rnn, axis=1))[0]
print('rows with different nn lists', len(bad), 'of', len(nn))
setdiff = [i for i in bad if set(nn[i].tolist()) != set(rnn[i].tolist())]
print('different SETS', len(setdiff))
for i in setdiff[:5]:
    d = np.sum((pts[1][nn[i]] - pts[1][i])**2, 1); dr = np.sum((pts[1][rnn[i]] - pts[1][i])**2, 1)
    print(i, nn[i].tolist(), d.tolist()); print('   ', rnn[i].tolist(), dr.tolist())
big = np.where(np.abs(nor[1]-ref).max(1) > 1e-7)[0]
print('normals differing', len(big), 'of which nn-set differs', len(set(big) & set(setdiff)))
for i in big[:5]:
    if i in setdiff: continue
    P = pts[1][rnn[i]]; c = P.mean(0); w, V = np.linalg.eigh((P-c).T@(P-c)); print(i, 'eigs', w, 'gpu', nor[1][i], 'ref', ref[i])
