"""Solver parameter sweep: PCG iterations and solve-stage time.  python tools/tune_smoother.py case [json list of config dicts]"""
import os, sys, time, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, mgbx
from mgbx import solver, geometry as G, hierarchy as H, problem as P
case = sys.argv[1]
if case.startswith("q1c"):
    prob = P.assemble(H.amg(G.structured_box(3, int(case[3:]), k=1)), p=1.0); kw = dict(t=0.01)
else:
    prob = P.assemble(H.amg(G.subdivide(G.fem2d_P1(), int(case))), p=1.5); kw = {}
base = None
cfgs = json.load(open(sys.argv[2])) if len(sys.argv) > 2 else [dict(), dict(precond_fp32=1), dict(precond_fp32=1, smoother=0), dict(smoother=0)]
for cfg in cfgs:
    try:
        for rep in range(2):
            t0 = time.time(); sol = solver.mgb_solve(prob, config=cfg, **kw); dt = time.time() - t0
    except Exception as e:
        print(json.dumps({"cfg": cfg, "failed": repr(e)[:120]}), flush=True)
        continue
    st = sol["stats"]
    print(json.dumps({"cfg": cfg, "newton": int(sol["SOL_main"]["its"].sum()), "pcg_iters": st["pcg_iters"], "ms_solve": round(st["ms_solve"]), "ms_f2": round(st["ms_f2"]),
                      "wall_s": round(dt, 2), "z_sum": float(np.sum(sol["z"]))}), flush=True)
