"""Kernel micro-benchmark on the 980k-cell NACA0012 SA case: per-kernel device times for one or more
builds of libdab200 (used to compare launch-bound / layout variants).  python scripts/kbench.py [lib.so ...]"""
import os, sys, tempfile, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
from dafoam_b200 import cases
from dafoam_b200.pyDASolvers import pyDASolvers

libs = sys.argv[1:] or [None]
cells = int(os.environ.get("KB_CELLS", "980000"))
nk = int(os.environ.get("KB_NK", "1"))
nj = int(os.environ["KB_NJ"]) if os.environ.get("KB_NJ") else max(8, int(round((cells / nk / 2.0) ** 0.5 / 2.0)) * 2)
tile = os.environ.get("KB_TILE")
mesh = cases.naca0012_ogrid(ni=2 * nj, nj=nj, nk=nk, span=1.0 if nk > 1 else 0.1, tile=tuple(int(v) for v in tile.split("x")) if tile else None,
                            family_major=bool(int(os.environ.get("KB_FAMILY", "0"))),
                            bface_by_owner=bool(int(os.environ["KB_BFO"])) if os.environ.get("KB_BFO") else None)
d = tempfile.mkdtemp(prefix="dab_kb_")
cases.write_case(d, mesh, cases.default_bcs_naca(), binary=True)
for lib in libs:
    opts = dict(normalizeStates=dict(U=10.0, p=50.0, nuTilda=1e-3, phi=1.0))
    sol = pyDASolvers("DASimpleFoam -python", opts, caseDir=d, _lib_path=lib)
    n = sol.getNLocalAdjointStates()
    y = np.zeros(sol.getNLocalCells()); sol.getOFField("yWall", "scalar", y)
    sol.updateOFFields(cases.boundary_layer_state(mesh, y, noise=0.001))
    sol.benchSetVector(np.random.default_rng(4321).uniform(-1, 1, n))
    sol.benchDevice(0, 5)
    out = {}
    for name, which in (("product", 0), ("forward", 1), ("RevA", 2), ("RevB", 3), ("RevC", 4)):
        out[name] = round(sol.benchDevice(which, 30)[0], 4)
    out["cells"] = sol.getNLocalCells()
    out["GB_alg"] = round(sol.algorithmicBytes(0) / 1e9, 4)
    print(os.path.basename(lib or "libdab200.so"), out, flush=True)
    del sol
