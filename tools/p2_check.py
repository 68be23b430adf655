import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np, mgbx, mgb_oracle as O
from mgbx import solver, geometry as G, hierarchy as H, problem as P
prob = P.assemble(H.amg(G.subdivide(G.fem2d_P2(bubble=False), 4)), p=1.5)
so = O.mgb_solve(prob)
for cfg in (dict(), dict(dense_direct_max=0, coarse_max=40), dict(dense_direct_max=0, coarse_max=40, pcg_rtol=1e-11),
            dict(dense_direct_max=0, coarse_max=40, pcg_rtol=1e-13), dict(dense_direct_max=0, coarse_max=40, smoother=0)):
    sd = solver.mgb_solve(prob, config=cfg)
    e = np.linalg.norm(sd["z"] - so["z"]) / np.linalg.norm(so["z"])
    print(cfg, "rel z err %.2e" % e, "its", sd["SOL_main"]["its"].sum(axis=0).tolist(), "pcg", sd["stats"]["pcg_iters"], "obj rel %.2e" % (abs(sd["SOL_main"]["c_dot_Dz"][-1] - so["SOL_main"]["c_dot_Dz"][-1]) / abs(so["SOL_main"]["c_dot_Dz"][-1])), flush=True)
print("oracle its", so["SOL_main"]["its"].sum(axis=0).tolist())
