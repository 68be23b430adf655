"""CPU laboratory for pure P2 (fem2d_P2 without bubble, the slack in :broken_P1): what does the exact element-local elimination
of the slack leave for the V-cycle PCG?

Records the oracle's fine-level Newton systems of the main ramp (tools/smoother_lab.py record_systems), measures how far the slack
block is from diagonal (the corners carry zero weight and P_e is the identity on the midpoints, so it is diagonal), condenses the
slack exactly and runs the emulated V-cycle PCG (relative residual 1e-7, at most 400 iterations) on the reduced systems.
Test/tuning infrastructure: imports oracle/.

    python tools/pure_p2_lab.py 6 4       # level 6, every 4th recorded system
"""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for d in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tools")):
    sys.path.insert(0, d)
import scipy.sparse as sp

import mgbx  # noqa: F401
from mgbx import geometry as G, hierarchy as H, problem as P
from smoother_lab import VCycle, condense, pcg, record_systems, transfers


def main():
    L = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    every = int(sys.argv[2]) if len(sys.argv) > 2 else 4
    prob = P.assemble(H.amg(G.subdivide(G.fem2d_P2(bubble=False), L)), p=1.0)
    M = prob.M[0]
    t0 = time.time()
    seen = record_systems(prob, {}, every=every, cap=40)
    offs = M.var_offsets[-1]
    print("pure P2 L%d: u unknowns %d, slack %d, %d systems recorded in %.0f s" % (L, offs[1] - offs[0], offs[2] - offs[1], len(seen), time.time() - t0), flush=True)
    Ts = transfers(M)
    for Hm, g, tc in seen:
        Hss = Hm[offs[1]:, offs[1]:].tocsr()
        d = Hss.diagonal()
        offd = abs(Hss - sp.diags(d)).sum() / abs(d).sum()
        S, gs = condense(Hm, g, M)
        its = []
        for opt in (dict(smoother="cheb", nu=2, ratio=8.0), dict(smoother="l1", nu=2)):
            try:
                its.append(pcg(S, gs, VCycle(S, Ts, **opt), rtol=1e-7, maxit=400))
            except Exception as e:
                its.append(repr(e)[:40])
        print("t*max|f| %-9.3g slack block off-diagonal (relative) %.1e  PCG its (cheb2 shipped, l1-Jacobi 2) %s" % (tc, offd, its), flush=True)


if __name__ == "__main__":
    main()
