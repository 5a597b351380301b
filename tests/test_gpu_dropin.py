"""The drop-in boundary (SURVEY 8b) end to end: the reference's OWN class declarations (EnergyFunctional.h, Residuals.h,
AccumulatedTopHessian.h, AccumulatedSCHessian.h, FrameHessian.h, PointHessian.h ...) with the product's forwarding translation units
(ldso_b200/host/dropin/dropin_backend.cc) in place of the reference's EnergyFunctional.cc / Residuals.cc / Accumulated*Hessian.cc,
driven by the restated FullSystem::optimize loop of oracle/ref_pin/ref_bench.cc -- the SAME driver and C interface as
oracle/_ref/libref_ba.so, which runs the reference's own translation units on the CPU. Same window in, same trajectory out.
What libref_ba.so computed is stored in tests/golden/reference_small.npz; the drop-in library compiles against an LDSO source tree's
headers (`make -C oracle ref_pin dropin REF=<tree>`) and travels as a file."""
import os

import numpy as np
import pytest

from tests import oracle_py
from tests.golden import make_golden

pytestmark = pytest.mark.gpu

needs_libs = pytest.mark.skipif(not os.path.exists(oracle_py.DROPIN_LIB),
                                reason="oracle/_ref/libdropin_ba.so compiles against an LDSO source tree's headers (make -C oracle ref_pin dropin REF=<tree>)")


@needs_libs
@pytest.mark.parametrize("which", ["small", "cfg2"])
def test_dropin_walks_the_reference_trajectory(which):
    win = make_golden.ref_window(which)
    gpu = oracle_py.RefBA(win, multithreaded=True, lib_path=oracle_py.DROPIN_LIB)      # reference classes, device back end, 6 caller threads
    g = oracle_py.reference_golden()                                                    # reference classes, reference back end, 1 thread
    energies_r = g[which + "_energy"]
    eg, er = gpu.optimize_begin(), energies_r[0]
    assert abs(eg - er) <= 1e-5 * abs(er), (eg, er)
    energies_g = [eg]
    for it in range(make_golden.TRAJECTORY_ITERATIONS):
        gpu.gn_iteration(it)
        energies_g.append(gpu.energy())
        if it == 0:
            # the first update off the gauge direction (the oracle's projector for this window: same evaluation points)
            P = oracle_py.OracleBA(win, threads_mode=1).nullspace_projector()
            I = np.eye(P.shape[0])
            xg, xr = gpu.last_x(), g[which + "_lastX0"]
            err = np.linalg.norm((I - P) @ (xg - xr)) / np.linalg.norm((I - P) @ xr)
            assert err < 1e-4, err
    # later iterates differ along the (noise-driven) gauge direction; energies and depths do not care
    assert np.allclose(energies_g, energies_r, rtol=2e-3), (energies_g, energies_r)
    assert energies_g[-1] < 0.5 * energies_g[0]
    idg, idr = gpu.idepths(), g[which + "_idepth"][-1]
    assert np.quantile(np.abs(idg - idr) / np.maximum(np.abs(idr), 1e-3), 0.99) < 1e-2


@needs_libs
def test_dropin_coarse_tracker_matches_reference():
    """CoarseTracker(w, h) / makeK / setCoarseTrackingRef / trackNewestCoarse of the reference's class declaration
    (include/frontend/CoarseTracker.h) with the product's dropin_tracker.cc, against the reference's own CoarseTracker.cc."""
    pair = make_golden.ref_track_pair("small")
    g = oracle_py.RefTracker(pair, lib_path=oracle_py.DROPIN_LIB).track(np.eye(3), np.zeros(3), 0.0, 0.0, pair.levels - 1)
    gold = oracle_py.reference_golden()
    r = (bool(gold["track_small_ok"]), gold["track_small_R"], gold["track_small_t"], *gold["track_small_aff"])
    assert g[0] == r[0]
    assert np.linalg.norm(g[1] - r[1]) < 1e-6 and np.linalg.norm(g[2] - r[2]) <= 1e-4 * np.linalg.norm(r[2])
    assert abs(g[3] - r[3]) < 1e-5 and abs(g[4] - r[4]) < 1e-3
