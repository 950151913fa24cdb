"""Kernel functors (compiled for the host: tests/hostsim, TEST-ONLY) vs the oracle.  This is how the
hand-derived reverse sweep is checked on a machine without a GPU; the -m gpu tests repeat the same
checks through the CUDA library."""
import numpy as np

from tests.common import HOSTSIM, check_functions, check_parity, setup, rel_err


def test_forward_and_reverse_parity_host_build():
    worst = check_parity(HOSTSIM, tol=1e-10)
    assert worst < 1e-10


def test_force_function_and_dfdw_host_build():
    dirv = [float(np.cos(0.05)), float(np.sin(0.05)), 0.0]
    fn = {"CD": {"type": "force", "source": "patchToFace", "patches": ["wing"], "directionMode": "fixedDirection",
                 "direction": dirv, "scale": 0.02}}
    mesh, bcs, orc, sol, W, _ = setup("naca", True, lib_path=HOSTSIM, extra_options=dict(function=fn))
    sol.updateOFFields(W)
    F, Fo = sol.calcFunction("CD"), orc.force(W, 0, dirv, 0.02)
    assert abs(F - Fo) <= 1e-12 * abs(Fo)
    prod = np.zeros(orc.ndof)
    sol.calcJacTVecProduct("states", "stateVar", W, "CD", "function", np.array([1.0]), prod)
    assert rel_err(prod, orc.dforce_dw(W, 0, dirv, 0.02)) < 1e-12


def test_force_moment_and_direction_modes_host_build():
    assert check_functions(HOSTSIM)


def test_dot_product_identity_host_build():
    # <J^T psi, v> == <psi, J v> with J v from central differences of the engine's own R(W)
    mesh, bcs, orc, sol, W, _ = setup("channel", True, lib_path=HOSTSIM, nk=1,
                                      extra_options=dict(normalizeStates=dict(U=1.0, p=1.0, nuTilda=1.0, phi=1.0)))
    sol.updateOFFields(W)
    rng = np.random.default_rng(5)
    n = orc.ndof
    psi = rng.uniform(-1, 1, n)
    y = np.zeros(n)
    sol.calcdRdWTPsiAD(psi, y)
    magSf = orc.geometry("magSf")
    y[-mesh.n_faces:] /= magSf  # undo the phi scaling (normalizeStates phi * magSf)
    v = rng.uniform(-1, 1, n) * 1e-3
    eps = 1e-4
    Rp, Rm = np.zeros(n), np.zeros(n)
    sol.updateOFFields(W + eps * v)
    sol.getResiduals(Rp)
    sol.updateOFFields(W - eps * v)
    sol.getResiduals(Rm)
    Jv = (Rp - Rm) / (2 * eps)
    assert abs(psi @ Jv - v @ y) <= 1e-6 * abs(v @ y)


def test_phi_rows_are_scaled_only_when_phi_is_listed_in_normalize_states():
    """DASolver::normalizeGradientVec (DASolver.C:2431-2452) multiplies the phi rows of a product by normalizeStates.phi * |Sf| only if
    "phi" is a key of normalizeStates; otherwise they are left alone (ADVICE round 1)."""
    ns = dict(U=10.0, p=50.0, nuTilda=1e-3)  # no phi
    from oracle.pyoracle import Oracle
    mesh, bcs, orc, sol, W, _ = setup("channel", True, nk=1, lib_path=HOSTSIM, extra_options=dict(normalizeStates=ns))
    orc2 = Oracle(mesh, bcs, normalizeStates=ns, divU="linearUpwind")
    sol.updateOFFields(W)
    orc2.record(W)
    psi = np.random.default_rng(9).uniform(-1, 1, orc2.ndof)
    y = np.zeros(orc2.ndof)
    sol.calcdRdWTPsiAD(psi, y)
    yo = orc2.jtvec(psi)
    assert rel_err(y, yo) < 1e-10
    # and it differs from the listed case by exactly |Sf| on the phi rows
    orc.record(W)
    y1 = orc.jtvec(psi)
    nF = mesh.n_faces
    assert rel_err(y1[-nF:], yo[-nF:] * orc.geometry("magSf")) < 1e-12


def test_reverse_parity_on_tile_major_ogrid_wing_prism_and_laminar_channel_host_build():
    """dRdW^T psi against the oracle on a 64x48 O-grid numbered tile by tile (16x12 tiles; linearUpwindV + wall function) and on
    the wing, prism and laminar channel meshes."""
    from tests.test_gpu_parity import _medium_case
    worst = 0.0
    mesh, orc, sol, W = _medium_case(64, 48, lib=HOSTSIM)
    sol.updateOFFields(W)
    orc.record(W)
    psi = np.random.default_rng(3).uniform(-1, 1, orc.ndof)
    y = np.zeros(orc.ndof)
    sol.calcdRdWTPsiAD(psi, y)
    worst = max(worst, rel_err(y, orc.jtvec(psi)))
    for kind, turb, nk in (("wing", True, 3), ("prism", True, 1), ("channel", False, 1)):
        mesh, bcs, orc, sol, W, _ = setup(kind, turb, nk=nk, lib_path=HOSTSIM)
        sol.updateOFFields(W)
        orc.record(W)
        psi = np.random.default_rng(3).uniform(-1, 1, orc.ndof)
        y = np.zeros(orc.ndof)
        sol.calcdRdWTPsiAD(psi, y)
        worst = max(worst, rel_err(y, orc.jtvec(psi)))
    assert worst < 1e-10, worst
