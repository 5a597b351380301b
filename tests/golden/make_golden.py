"""Generate the frozen oracle outputs used by tests/test_oracle_cpu.py and the GPU parity tests.

    python tests/golden/make_golden.py
The inputs are the seeded synthetic windows of ldso_b200.synth; the outputs come from oracle/liboracle.so
(-ffp-contract=off build, serial emulation of the reference's 6 worker accumulators).
The reference itself ships no golden vectors for this path (SURVEY.md §4).

    python tests/golden/make_golden.py --reference
writes reference_small.npz: what the reference's own translation units compute on the cases of the tests that compare with
the reference (oracle/_ref/libref_ba.so, built by `make -C oracle ref_pin REF=<LDSO source tree>`), so that those tests
run without the reference sources.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from ldso_b200 import synth  # noqa: E402
from tests import oracle_py  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    win = synth.make_window(nF=5, pts_per_frame=60, w=320, h=240, seed=3)
    o = oracle_py.OracleBA(win, threads_mode=0)
    e0 = o.optimize_begin()
    o.solve_system(0)
    s = o.system()
    r = o.residuals()
    p = o.points()
    P = o.nullspace_projector()
    np.savez_compressed(os.path.join(HERE, "ba_small.npz"), energy0=e0, HA=s["HA"], bA=s["bA"], Hsc=s["Hsc"], bsc=s["bsc"],
                        lastHS=s["lastHS"], lastbS=s["lastbS"], lastX=s["lastX"], P=P, state_NewState=r["state_NewState"],
                        J=r["J"], JpJdF=r["JpJdF"], isActive=r["isActive"], HdiF=p["HdiF"], bdSumF=p["bdSumF"], step=p["step"])
    pair = synth.make_track_pair(w=320, h=240, n_pts=400, seed=7)
    ot = oracle_py.OracleTracker(pair)
    res, H, b = ot.eval(0, np.eye(3), np.zeros(3), 0.0, 0.0, 20.0)
    ok, R, t, a, bb, lr, lf, ne = ot.track(np.eye(3), np.zeros(3), 0.0, 0.0, pair.levels - 1)
    np.savez_compressed(os.path.join(HERE, "tracker_small.npz"), res0=res, H0=H, b0=b, R=R, t=t, aff=np.array([a, bb]), lastResiduals=lr,
                        lastFlow=lf, n_evals=ne)
    # immature-point trace: two traceNewCoarse passes over 150 candidates per host keyframe
    wt = synth.make_window(nF=6, pts_per_frame=10, w=320, h=240, seed=3)
    case = synth.make_trace_case(wt, 150, seed=5)
    tr = oracle_py.OracleTrace(wt, case)
    st1 = tr.trace_on(wt.nF - 2)
    imin1, imax1 = tr.idepth_min.copy(), tr.idepth_max.copy()
    st2 = tr.trace_on(wt.nF - 1)
    np.savez_compressed(os.path.join(HERE, "trace_small.npz"), color=tr.color, weights=tr.weights, gradH=tr.gradH, status1=st1, status2=st2,
                        idepth_min1=imin1, idepth_max1=imax1, idepth_min2=tr.idepth_min, idepth_max2=tr.idepth_max, quality=tr.quality,
                        uv=tr.uv, interval=tr.interval)
    make_select()
    print("golden written")


def select_case():
    """The activation-selection case shared by make_select() and the tests: window, traced candidates, arguments."""
    win = synth.make_window(nF=6, pts_per_frame=40, w=320, h=240, seed=3)
    case = synth.make_trace_case(win, 300, seed=5)
    tr = oracle_py.OracleTrace(win, case)
    tr.trace_on(win.nF - 2)
    tr.trace_on(win.nF - 1)
    newest = win.nF - 1
    m = case.host != newest
    n = int(m.sum())
    my_type = np.random.default_rng(11).choice(np.array([1.0, 2.0, 4.0], np.float32), n)
    quality = np.where(np.isfinite(tr.quality[m]), tr.quality[m], 0).astype(np.float32)
    flagged = np.zeros(win.nF, np.uint8)
    flagged[0] = 1
    args = (case.u[m], case.v[m], case.host[m], tr.idepth_min[m], tr.idepth_max[m], tr.status[m], tr.interval[m], quality, my_type)
    return win, newest, args, flagged


def make_select():
    # activatePointsMT's selection: actions and the level-1 distance map for two minimum distances
    win, newest, args, flagged = select_case()
    o = oracle_py.OracleBA(win, threads_mode=0)
    a13, m13 = o.select_activation(newest, 1.3, *args, frame_flagged=flagged)
    a20, m20 = o.select_activation(newest, 2.0, *args, frame_flagged=flagged)
    _, m0 = o.select_activation(newest, 2.0, *(x[:0] for x in args), frame_flagged=flagged)
    np.savez_compressed(os.path.join(HERE, "select_small.npz"), action13=a13, map13=m13.astype(np.uint16), action20=a20, map20=m20.astype(np.uint16),
                        map_seed_only=m0.astype(np.uint16))


# The cases of the tests that compare with the reference. make_reference() and those tests both build them from here.
def ref_window(name):
    """small: test_reference_arm_matches_oracle, test_dropin_walks_the_reference_trajectory[small]; cfg2: the same test's [cfg2];
    gauge: test_reference_lastx_noise_floor_is_along_the_gauge; bookkeeping: test_dropin_bookkeeping_matches_reference."""
    return {"small": lambda: synth.make_window(nF=5, pts_per_frame=60, w=320, h=240, seed=3),
            "cfg2": lambda: synth.make_window(nF=8, pts_per_frame=250, seed=42),
            "gauge": lambda: synth.make_window(nF=6, pts_per_frame=120, w=320, h=240, seed=17),
            "bookkeeping": lambda: synth.make_window(nF=5, pts_per_frame=30, w=320, h=240, seed=5)}[name]()


def ref_track_pair(name):
    """full: test_reference_tracker_matches_oracle; small: test_dropin_coarse_tracker_matches_reference."""
    return synth.make_track_pair() if name == "full" else synth.make_track_pair(w=320, h=240, n_pts=400, seed=7)


TRAJECTORY_ITERATIONS = 5       # Gauss-Newton iterations stored for the small and cfg2 windows
BOOKKEEPING_CASES = [(-1, 0), (1, 7), (4, 3)]
MAKE_K_GEOMETRIES = [(640, 480, 4, (400.0, 400.0, 319.5, 239.5)), (1232, 368, 5, (718.856, 718.856, 607.1928, 185.2157))]


def _ref_trajectory(out, key, win, iterations, multithreaded=False):
    """Energies after optimize's prologue and after each Gauss-Newton iteration, the step-size criteria, the first update and the
    inverse depths after each iteration of the reference's back end on `win`."""
    r = oracle_py.RefBA(win, multithreaded=multithreaded)
    energies, converged, idepths = [r.optimize_begin()], [], []
    for it in range(iterations):
        converged.append(r.gn_iteration(it))
        energies.append(r.energy())
        idepths.append(r.idepths())
        if it == 0:
            out[key + "_lastX0"] = r.last_x()
    out[key + "_energy"] = np.array(energies)
    out[key + "_converged"] = np.array(converged)
    out[key + "_idepth"] = np.array(idepths)


def make_reference():
    import ctypes as C
    if oracle_py.ref_lib() is None:
        raise SystemExit("oracle/_ref/libref_ba.so is not built: make -C oracle ref_pin REF=<LDSO source tree>")
    out = {}
    small = ref_window("small")
    _ref_trajectory(out, "small", small, TRAJECTORY_ITERATIONS)
    _ref_trajectory(out, "small_6threads", small, 1, multithreaded=True)
    _ref_trajectory(out, "cfg2", ref_window("cfg2"), TRAJECTORY_ITERATIONS)
    gauge = ref_window("gauge")
    _ref_trajectory(out, "gauge", gauge, 1)
    _ref_trajectory(out, "gauge_6threads", gauge, 1, multithreaded=True)
    for name in ("full", "small"):
        pair = ref_track_pair(name)
        ok, R, t, a, b, _ = oracle_py.RefTracker(pair).track(np.eye(3), np.zeros(3), 0.0, 0.0, pair.levels - 1)
        key = "track_" + name
        out[key + "_ok"], out[key + "_R"], out[key + "_t"], out[key + "_aff"] = ok, R, t, np.array([a, b])
    # EnergyFunctional's bookkeeping under scripted window maintenance
    bk = ref_window("bookkeeping")
    for drop_target, remove_every in BOOKKEEPING_CASES:
        r = oracle_py.RefBA(bk, multithreaded=False)
        buf = (C.c_longlong * 20000)()
        r.L.ref_ba_bookkeeping.restype = C.c_int
        n = r.L.ref_ba_bookkeeping(r.o, drop_target, remove_every, buf, 20000)
        assert 0 < n <= 20000
        out[f"bookkeeping_{drop_target}_{remove_every}"] = np.array(buf[:n], np.int64)
    # CoarseTracker(w, h) + makeK
    L = oracle_py.ref_lib()
    L.ref_tracker_make_k.restype = C.c_int
    for w, h, levels, K in MAKE_K_GEOMETRIES:
        k = np.zeros(10 * levels)
        assert L.ref_tracker_make_k(w, h, levels, np.array(K, np.float64).ctypes.data_as(C.POINTER(C.c_double)),
                                    k.ctypes.data_as(C.POINTER(C.c_double))) == levels
        out[f"make_k_{w}x{h}"] = k
    np.savez_compressed(os.path.join(HERE, "reference_small.npz"), **out)


if __name__ == "__main__":
    if "--reference" in sys.argv:
        make_reference()
    else:
        main()
