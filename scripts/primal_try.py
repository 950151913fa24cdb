"""Development driver: SIMPLE primal on a small case with the host-simulation build."""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.common import setup, HOSTSIM

kind = sys.argv[1] if len(sys.argv) > 1 else "channel"
scale = int(sys.argv[2]) if len(sys.argv) > 2 else 1
iters = int(sys.argv[3]) if len(sys.argv) > 3 else 300
mesh, bcs, orc, sol, W, d = setup(kind, True, lib_path=HOSTSIM, nk=1, scale=scale, with_oracle=False,
                                  extra_options=dict(primalMaxIters=iters, primalMinResTol=1e-9, printInterval=20,
                                                     adjEqnOption=dict(printInfo=1)))
n = sol.getNLocalAdjointStates()
R = np.zeros(n)
sol.getResiduals(R)
print("cells", mesh.n_cells, "|R0|", np.linalg.norm(R))
t = time.time()
fail = sol.solvePrimal()
st = sol.primalStats
print("fail", fail, "iters", st.iterations, "maxRes", st.max_residual, "pIters", st.p_iterations, "sec", time.time() - t)
sol.getResiduals(R)
print("|R|", np.linalg.norm(R), np.abs(R).max())
W = np.zeros(n); sol.getOFFields(W)
nC = mesh.n_cells
print("U range", W[:3*nC].reshape(-1,3).min(0), W[:3*nC].reshape(-1,3).max(0), "p", W[3*nC:4*nC].min(), W[3*nC:4*nC].max(), "nt", W[4*nC:5*nC].min(), W[4*nC:5*nC].max())
