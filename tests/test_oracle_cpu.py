"""CPU tests of the oracle (the parity checker) and of the synthetic-input builder. No GPU needed.

The reference ships no golden vectors for this path and its build cannot run here. What pins the oracle: (0) nine of the reference's
own translation units (Residuals.cc, ImmaturePoint.cc, PointHessian.cc, FrameHessian.cc, FrameFramePrecalc.cc, AccumulatedTopHessian.cc,
AccumulatedSCHessian.cc, EnergyFunctional.cc, CoarseTracker.cc) and their headers are compiled from its sources against stand-in
Eigen / Sophus headers and compared bit for bit (oracle/ref_pin, test_oracle_pinned_against_reference_sources); for Eigen / Sophus
themselves and the FullSystem driver loop (1) independent re-derivations of the same algebra in double-precision numpy, (2) invariants the algorithm must
satisfy, (3) frozen outputs in tests/golden/.
"""
import os

import numpy as np
import pytest

from ldso_b200 import synth
from tests import oracle_py
from tests.golden import make_golden
from tests.parity import rel_err

GOLD = os.path.join(os.path.dirname(__file__), "golden", "ba_small.npz")


@pytest.fixture(scope="module")
def small_win():
    return synth.make_window(nF=5, pts_per_frame=60, w=320, h=240, seed=3)


@pytest.fixture(scope="module")
def solved(small_win):
    o = oracle_py.OracleBA(small_win, threads_mode=0)
    e0 = o.optimize_begin()
    o.solve_system(0)
    return o, e0


def test_make_images_matches_numpy(small_win):
    color = small_win.pyramids[2][0][:, :, 0]
    om = oracle_py.make_images(color, small_win.levels)
    for l in range(small_win.levels):
        assert np.array_equal(om[l], small_win.pyramids[2][l])


def test_se3_exp_log_roundtrip():
    from scipy.spatial.transform import Rotation
    import ctypes as C
    L = oracle_py.lib()
    rng = np.random.default_rng(0)
    for _ in range(20):
        a = rng.normal(0, 0.3, 6)
        R = np.zeros(9); t = np.zeros(3); back = np.zeros(6)
        L.oracle_se3_exp(a.ctypes.data_as(oracle_py.c_dp), R.ctypes.data_as(oracle_py.c_dp), t.ctypes.data_as(oracle_py.c_dp))
        assert np.allclose(R.reshape(3, 3), Rotation.from_rotvec(a[3:]).as_matrix(), atol=1e-12)
        L.oracle_se3_log(R.ctypes.data_as(oracle_py.c_dp), t.ctypes.data_as(oracle_py.c_dp), back.ctypes.data_as(oracle_py.c_dp))
        assert np.allclose(back, a, atol=1e-10)


def test_ldlt_solve_matches_numpy():
    L = oracle_py.lib()
    rng = np.random.default_rng(1)
    n = 68
    M = rng.normal(size=(n, n))
    A = M @ M.T + np.diag(rng.uniform(0, 1e3, n))
    b = rng.normal(size=n)
    x = np.zeros(n)
    Af = np.asfortranarray(A)
    L.oracle_ldlt_solve(n, Af.ctypes.data_as(oracle_py.c_dp), b.ctypes.data_as(oracle_py.c_dp), x.ctypes.data_as(oracle_py.c_dp))
    assert rel_err(x, np.linalg.solve(A, b)) < 1e-9


def test_states_and_counts(solved, small_win):
    o, e0 = solved
    r = o.residuals()
    assert e0 > 0
    assert r["isActive"].sum() == (r["state_state"] == 0).sum()
    assert o.res_counts()[0] == r["isActive"].sum()
    # OOB residuals never become active and report energy -1
    assert np.all(r["state_NewEnergyWithOutlier"][r["state_NewState"] == 1] == -1)


def test_HA_symmetric_Hsc_nearly(solved):
    o, _ = solved
    s = o.system()
    assert np.abs(s["HA"] - s["HA"].T).max() <= 1e-12 * np.abs(s["HA"]).max()
    assert np.abs(s["Hsc"] - s["Hsc"].T).max() <= 1e-6 * np.abs(s["Hsc"]).max()


def _absolute_rows(o, win):
    """Independent double-precision re-derivation: map every active residual's relative Jacobian rows into the
    68-dim absolute state through the adjoints and return per-point w_p, Hdd, bd (numpy, float64)."""
    r = o.residuals()
    f = o.frames()
    nF = win.nF
    n = 8 * nF + 4
    rp = win.res_point
    J = r["J"].astype(np.float64)
    per_point = {}
    HA = np.zeros((n, n)); bA = np.zeros(n)
    for k in range(win.nR):
        if not r["isActive"][k]:
            continue
        h = int(win.pt_host[rp[k]]); t = int(win.res_target[k])
        AH = f["adHost"][h + nF * t]; AT = f["adTarget"][h + nF * t]
        G = np.zeros((12, n))                       # [C(4) | rel(8)] -> absolute
        G[0:4, 0:4] = np.eye(4)
        G[4:12, 4 + 8 * h:12 + 8 * h] = AH.T
        G[4:12, 4 + 8 * t:12 + 8 * t] = AT.T
        resF = J[k, 0:8]; Jpdxi = J[k, 8:20].reshape(2, 6); Jpdc = J[k, 20:28].reshape(2, 4); Jpdd = J[k, 28:30]
        JIdx = J[k, 30:46].reshape(2, 8); JabF = J[k, 46:62].reshape(2, 8)
        # per-pixel row in [C | xi | ab] coordinates
        rows = np.zeros((8, 12))
        rows[:, 0:4] = JIdx[0][:, None] * Jpdc[0][None, :] + JIdx[1][:, None] * Jpdc[1][None, :]
        rows[:, 4:10] = JIdx[0][:, None] * Jpdxi[0][None, :] + JIdx[1][:, None] * Jpdxi[1][None, :]
        rows[:, 10] = JabF[0]; rows[:, 11] = JabF[1]
        Ja = rows @ G                               # 8 x n
        jd = JIdx[0] * Jpdd[0] + JIdx[1] * Jpdd[1]  # 8, d r / d idepth
        HA += Ja.T @ Ja
        bA += Ja.T @ resF
        pp = per_point.setdefault(int(rp[k]), dict(w=np.zeros(n), Hdd=0.0, bd=0.0))
        pp["w"] += Ja.T @ jd
        pp["Hdd"] += jd @ jd
        pp["bd"] += jd @ resF
    return HA, bA, per_point


def test_accumulate_and_stitch_against_numpy(solved, small_win):
    """H_A, b_A, H_sc, b_sc of the oracle == direct absolute-coordinate accumulation in float64 numpy."""
    o, _ = solved
    s = o.system()
    HA, bA, per_point = _absolute_rows(o, small_win)
    n = HA.shape[0]
    Hsc = np.zeros((n, n)); bsc = np.zeros(n)
    for pp in per_point.values():
        Hd = max(pp["Hdd"], 1e-10)
        Hsc += np.outer(pp["w"], pp["w"]) / Hd
        bsc += pp["w"] * pp["bd"] / Hd
    assert rel_err(s["HA"], HA) < 2e-5
    assert rel_err(s["bA"], bA) < 2e-5
    assert rel_err(s["Hsc"], Hsc) < 2e-5
    assert rel_err(s["bsc"], bsc) < 2e-5


def test_solution_satisfies_system(solved):
    o, _ = solved
    s = o.system()
    n = s["lastHS"].shape[0]
    lam = 1e-5
    Hf = s["lastHS"] + s["Hsc"]
    H2 = Hf.copy(); H2[np.diag_indices(n)] *= (1 + lam); H2 -= s["Hsc"] / (1 + lam)
    res = H2 @ s["lastX"] - s["lastbS"]
    assert np.linalg.norm(res) <= 1e-6 * np.linalg.norm(s["lastbS"])


def test_zero_residual_for_identical_frames():
    """Two keyframes with the same pose, image and affine parameters: every residual is 0, so energy and b vanish."""
    win = synth.make_window(nF=2, pts_per_frame=40, w=320, h=240, seed=5, outlier_frac=0.0)
    win.Rcw[1] = win.Rcw[0]; win.tcw[1] = win.tcw[0]
    win.pyramids[1] = win.pyramids[0]
    win.state_zero[:] = 0; win.state[:] = 0
    win.pt_idepth[:] = win.pt_idepth_zero
    # colours of points hosted in frame 1 were sampled from the old frame-1 image: resample from frame 0's
    for p in range(win.nP):
        for k in range(8):
            c, gx, gy = synth.sample_bilin(win.pyramids[0][0], np.array([win.pt_u[p] + synth.PATTERN[k, 0]]), np.array([win.pt_v[p] + synth.PATTERN[k, 1]]))
            win.pt_color[p, k] = c[0]
    o = oracle_py.OracleBA(win, threads_mode=1)
    e = o.optimize_begin()
    assert e < 1e-3
    o.solve_system(0)
    s = o.system()
    assert np.linalg.norm(s["bA"]) < 1e-2 * max(1.0, np.linalg.norm(np.diag(s["HA"]))) * 1e-3


def test_gn_decreases_energy(small_win):
    o = oracle_py.OracleBA(small_win, threads_mode=1)
    e = [o.optimize_begin()]
    for it in range(4):
        o.gn_iteration(it)
        e.append(o.L.oracle_ba_last_energy(o.o))
    assert e[-1] < 0.2 * e[0]
    # idepths move towards the truth
    err0 = np.median(np.abs(small_win.pt_idepth - small_win.pt_idepth_true))
    err1 = np.median(np.abs(o.points()["idepth"] - small_win.pt_idepth_true))
    assert err1 < err0


def test_thread_modes_agree_up_to_gauge(small_win):
    """6-way split accumulation vs a single accumulator: pieces agree to float rounding; the raw update vector does
    NOT (the scale gauge is only damped by lambda=1e-5), its gauge-orthogonal part does. This is the reference's own
    run-to-run noise floor and the reason parity on lastX is measured after projecting out the null space."""
    res = {}
    for mode in (0, 1):
        o = oracle_py.OracleBA(small_win, threads_mode=mode)
        o.optimize_begin()
        o.solve_system(0)
        res[mode] = o.system()
        P = o.nullspace_projector()
    for k in ("HA", "bA", "Hsc", "bsc"):
        assert rel_err(res[1][k], res[0][k]) < 1e-6
    I = np.eye(P.shape[0])
    assert rel_err((I - P) @ res[1]["lastX"], (I - P) @ res[0]["lastX"]) < 1e-4


def test_golden_small_window(small_win):
    """Frozen oracle outputs (tests/golden/make_golden.py). Guards the checker itself against silent edits."""
    assert os.path.exists(GOLD), "run python tests/golden/make_golden.py"
    g = np.load(GOLD)
    o = oracle_py.OracleBA(small_win, threads_mode=0)
    e0 = o.optimize_begin()
    o.solve_system(0)
    s = o.system()
    assert abs(e0 - float(g["energy0"])) <= 1e-9 * abs(e0)
    for k in ("HA", "bA", "Hsc", "bsc", "lastHS", "lastbS"):
        assert rel_err(s[k], g[k]) < 1e-9, k
    r = o.residuals()
    assert np.array_equal(r["state_NewState"], g["state_NewState"])
    assert rel_err(r["J"], g["J"]) < 1e-7


def test_tracker_converges_to_truth():
    pair = synth.make_track_pair(w=320, h=240, n_pts=400, seed=7)
    ot = oracle_py.OracleTracker(pair)
    ok, R, t, a, b, lr, lf, ne = ot.track(np.eye(3), np.zeros(3), 0.0, 0.0, pair.levels - 1)
    assert ok
    assert np.linalg.norm(t - pair.t_true) < 0.1 * np.linalg.norm(pair.t_true)
    assert np.abs(R - pair.R_true).max() < 2e-3
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "tracker_small.npz"))
    assert rel_err(t, g["t"]) < 1e-9 and rel_err(R, g["R"]) < 1e-9
    res, H, bb = ot.eval(0, np.eye(3), np.zeros(3), 0.0, 0.0, 20.0)
    assert rel_err(H, g["H0"]) < 1e-9 and rel_err(bb, g["b0"]) < 1e-9 and rel_err(res, g["res0"]) < 1e-9


def test_marginalize_frame_prior():
    """EnergyFunctional::marginalizeFrame's HM/bM algebra (EnergyFunctional.cc:72-129) against an independent numpy
    derivation, and the defining property of a Schur complement: the kept variables of the full solution solve the
    reduced system."""
    win = synth.make_window(nF=5, pts_per_frame=40, w=320, h=240, seed=3)
    n = 8 * win.nF + 4
    rng = np.random.default_rng(17)
    B = rng.standard_normal((n, n)) * np.exp(rng.uniform(0, 6, n))[:, None]
    HM = B @ B.T + np.diag(rng.uniform(1, 100, n))
    bM = rng.standard_normal(n) * 100.0
    for idx in (0, 2, win.nF - 1):
        o = oracle_py.OracleBA(win, threads_mode=1)
        o.set_marg_prior(HM, bM)
        fr = o.frames()
        prior, dprior = fr["prior"][idx], fr["delta_prior"][idx]
        Hn, bn = o.marginalize_frame(idx)
        nd = n - 8
        assert Hn.shape == (nd, nd)
        io = 4 + 8 * idx
        keep = np.r_[0:io, io + 8:n]
        p = np.r_[keep, io:io + 8]
        H = HM[np.ix_(p, p)].copy(); b = bM[p].copy()
        H[nd:, nd:] += np.diag(prior); b[nd:] += prior * dprior
        S = np.sqrt(np.abs(np.diag(H)) + 10.0)
        Hs = H / S[:, None] / S[None, :]; bs = b / S
        hpi = np.linalg.inv(Hs[nd:, nd:])
        bli = Hs[nd:, :nd].T @ hpi
        Ht = Hs[:nd, :nd] - bli @ Hs[nd:, :nd]
        bt = bs[:nd] - bli @ bs[nd:]
        Ht = Ht * S[:nd, None] * S[None, :nd]; bt = bt * S[:nd]
        Ht = 0.5 * (Ht + Ht.T)
        assert rel_err(Hn, Ht) < 1e-9 and rel_err(bn, bt) < 1e-9
        assert np.array_equal(Hn, Hn.T)
        x_full = np.linalg.solve(H, b)
        assert rel_err(np.linalg.solve(Hn, bn), x_full[:nd]) < 1e-6


def test_trace_immature_oracle():
    """ImmaturePoint construction + traceOn (oracle/trace.cc): frozen outputs, and what the search is for — after two traces the
    true inverse depth of a well-traced candidate lies inside its [idepth_min, idepth_max] interval."""
    win = synth.make_window(nF=6, pts_per_frame=10, w=320, h=240, seed=3)
    case = synth.make_trace_case(win, 150, seed=5)
    tr = oracle_py.OracleTrace(win, case)
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "trace_small.npz"))
    assert np.array_equal(tr.color, g["color"]) and np.array_equal(tr.gradH, g["gradH"])
    st1 = tr.trace_on(win.nF - 2)
    assert np.array_equal(st1, g["status1"])
    assert np.array_equal(tr.idepth_min, g["idepth_min1"]) and np.array_equal(tr.idepth_max, g["idepth_max1"], equal_nan=True)
    st2 = tr.trace_on(win.nF - 1)
    assert np.array_equal(st2, g["status2"]) and np.array_equal(tr.idepth_max, g["idepth_max2"], equal_nan=True)
    good = st2 == oracle_py.IPS_GOOD
    assert good.sum() > 0.4 * case.n
    idt = np.zeros(case.n)
    for h in np.unique(case.host):
        m = case.host == h
        _, _, depth, _ = synth.scene_depth(win.Rcw[h], win.tcw[h], win.K, case.u[m].astype(float), case.v[m].astype(float))
        idt[m] = 1.0 / depth
    inside = (tr.idepth_min <= idt) & (idt <= tr.idepth_max)
    assert inside[good].mean() > 0.8
    # a candidate that left the image stays out
    oob = st2 == oracle_py.IPS_OOB
    st3 = tr.trace_on(win.nF - 1)
    assert np.all(st3[oob] == oracle_py.IPS_OOB)


PIN_DIR = os.path.join(oracle_py.ORACLE_DIR, "_ref")


@pytest.mark.skipif(not all(os.path.exists(os.path.join(PIN_DIR, n)) for n in ("pin_ref", "pin_ref_break")),
                    reason="oracle/_ref/pin_ref compiles an LDSO source tree's own sources (build() makes it where the tree is present; "
                           "make -C oracle ref_pin REF=<tree>)")
def test_oracle_pinned_against_reference_sources():
    """oracle/ref_pin: the reference's OWN Residuals.cc (linearize, applyRes/takeData, fixLinearizationF), AccumulatedTopHessian.cc /
    AccumulatedSCHessian.cc (addPoint<0,1,2>, SC addPoint, the stitchers), EnergyFunctional.cc (insertFrame, setAdjointsF, setDeltaF,
    solveSystemF, resubstitute, orthogonalize, energies, marginalizePointsF, marginalizeFrame), FrameHessian.cc, FrameFramePrecalc.cc,
    PointHessian.cc, CoarseTracker.cc (makeK, makeCoarseDepthL0, calcRes, calcGSSSE, trackNewestCoarse), ImmaturePoint.cc (constructor,
    traceOn, linearizeResidual), MatrixAccumulators.h, GlobalFuncs.h, ResidualProjections.h, AffLight.h and Setting.cc, compiled
    unmodified where they lie (against oracle/ref_shim: stand-ins for Eigen / Sophus / Frame.h / OpenCV / glog), agree bit for bit
    with the oracle on 108 checks; the negative controls (an operand scaled by 1 + 2e-7, two results moved by one ulp on the oracle
    side) are detected. The two programs are the ones build() made (the reference's sources are needed to compile them, not to
    run them)."""
    import subprocess
    r = subprocess.run([os.path.join(PIN_DIR, "pin_ref")], capture_output=True, text=True)
    assert r.returncode == 0 and "PIN OK" in r.stdout, r.stdout + r.stderr
    r = subprocess.run([os.path.join(PIN_DIR, "pin_ref_break")], capture_output=True, text=True)
    assert r.returncode != 0 and "PIN MISMATCH" in r.stdout


def test_select_activation_oracle():
    """CoarseDistanceMap + activatePointsMT's selection (oracle): invariants of the greedy pass. (The map code itself is pinned against
    the reference's CoarseDistanceMap by oracle/ref_pin.)"""
    win = synth.make_window(nF=6, pts_per_frame=40, w=320, h=240, seed=3)
    case = synth.make_trace_case(win, 300, seed=5)
    tr = oracle_py.OracleTrace(win, case)
    tr.trace_on(win.nF - 2); tr.trace_on(win.nF - 1)
    newest = win.nF - 1
    m = case.host != newest
    n = int(m.sum())
    quality = np.where(np.isfinite(tr.quality[m]), tr.quality[m], 0).astype(np.float32)
    args = (case.u[m], case.v[m], case.host[m], tr.idepth_min[m], tr.idepth_max[m], tr.status[m], tr.interval[m], quality, np.ones(n, np.float32))
    o = oracle_py.OracleBA(win, threads_mode=0)
    _, base = o.select_activation(newest, 2.0, *(a[:0] for a in args))          # makeDistanceMap alone
    assert set(np.unique(base).tolist()) <= set(range(40)) | {1000} and (base == 0).sum() > 50
    prev = None
    for dist in (0.0, 1.0, 2.0, 4.0):
        act, dmap = o.select_activation(newest, dist, *args)
        assert set(np.unique(act).tolist()) <= {0, 1, 2}
        assert (dmap <= base).all()                                              # accepted points only ever shrink distances
        assert (dmap == 0).sum() - (base == 0).sum() <= (act == 1).sum()          # every new zero is an accepted candidate
        never = ~np.isfinite(tr.idepth_max[m]) | (tr.status[m] == oracle_py.IPS_OUTLIER)
        assert (act[never] == 2).all()
        if prev is not None:
            assert (act == 1).sum() <= prev                                       # a larger minimum distance accepts fewer
        prev = (act == 1).sum()
    assert prev > 0


def test_reference_arm_matches_oracle():
    """bench.py's reference arm (oracle/_ref/libref_ba.so: the reference's own back-end translation units + a restated FullSystem driver
    loop, built with -O3 -march=native) walks the same Gauss-Newton trajectory as the oracle port on the same window: energies, the
    step-size criterion and the final inverse depths agree up to the FMA-contraction noise of the two optimised builds. The reference's
    side is stored in tests/golden/reference_small.npz."""
    g = oracle_py.reference_golden()
    win = make_golden.ref_window("small")
    o = oracle_py.OracleBA(win, threads_mode=1, fast=True)
    e_r, e_o = g["small_energy"][0], o.optimize_begin()
    assert abs(e_r - e_o) <= 1e-6 * e_o
    for it in range(4):
        assert g["small_converged"][it] == o.gn_iteration(it)
        e_r = g["small_energy"][it + 1]
        assert abs(e_r - o.energy()) <= 2e-3 * e_r
    d = np.abs(g["small_idepth"][3] - o.points()["idepth"])
    assert np.median(d) < 3e-4 and d.max() < 5e-3          # the scale gauge is only damped (DESIGN section 5): a common drift of a few 1e-5
    # and with the reference's 6 worker threads (chunk sums arrive in thread order: compare loosely)
    e6 = g["small_6threads_energy"]
    assert abs(e6[0] - e_o) <= 1e-5 * e_o
    assert np.isfinite(e6[1]) and e6[1] < e_o


def test_reference_lastx_noise_floor_is_along_the_gauge():
    """Why parity on lastX is measured on the gauge-orthogonal complement: the reference's OWN library (its EnergyFunctional.cc, its
    accumulators, the stand-in Eigen's LDLT) and the oracle (same pinned H and b, Eigen's LDLT restated) give update vectors that differ
    by ~2e-3 as they stand -- twenty times the 1e-4 bar -- and by ~1e-5 once the seven gauge directions are projected out
    (measured: 1.6e-3 / 6.3e-6 on this window, 2.1e-3 / 1.2e-5 on the 8 x 2000-point window). Its 6-thread runs reproduced the
    1-thread bits in 5 of 5 runs on this host (the chunk scheduler hands one worker nearly everything), so the thread order is not
    the larger effect here; the factorisation's rounding along the barely-damped scale direction is. The reference's update vectors
    are stored in tests/golden/reference_small.npz."""
    g = oracle_py.reference_golden()
    win = make_golden.ref_window("gauge")
    xr = g["gauge_lastX0"]
    o = oracle_py.OracleBA(win, threads_mode=0)
    o.optimize_begin(); o.solve_system(0)
    xo = o.system()["lastX"]
    P = o.nullspace_projector()
    I = np.eye(P.shape[0])
    raw, proj = rel_err(xo, xr), rel_err((I - P) @ xo, (I - P) @ xr)
    assert proj < 1e-4, proj
    assert proj < 0.1 * raw or raw < 1e-5, (raw, proj)          # the disagreement lives in the gauge directions
    assert rel_err((I - P) @ g["gauge_6threads_lastX0"], (I - P) @ xr) < 1e-4


needs_dropin = pytest.mark.skipif(not os.path.exists(oracle_py.DROPIN_LIB),
                                  reason="oracle/_ref/libdropin_ba.so compiles against an LDSO source tree's headers (make -C oracle ref_pin dropin REF=<tree>)")


@needs_dropin
@pytest.mark.parametrize("drop_target,remove_every", make_golden.BOOKKEEPING_CASES)
def test_dropin_bookkeeping_matches_reference(drop_target, remove_every):
    """The drop-in translation units' HOST logic (ldso_b200/host/dropin: insertFrame / insertResidual / dropResidual / removePoint /
    makeIDX, the counters, the connectivity map, hostIDX / targetIDX) against the reference's own EnergyFunctional.cc, both driven through
    the reference's classes by the same scripted window maintenance (oracle/ref_pin/ref_bench.cc: ref_ba_bookkeeping; the reference's
    record is stored in tests/golden/reference_small.npz). No arithmetic member is called: the device context of the drop-in is created
    lazily, so this runs without a GPU."""
    import ctypes as C
    win = make_golden.ref_window("bookkeeping")
    got = {"ref": oracle_py.reference_golden()[f"bookkeeping_{drop_target}_{remove_every}"]}
    r = oracle_py.RefBA(win, multithreaded=False, lib_path=oracle_py.DROPIN_LIB)
    out = (C.c_longlong * 20000)()
    r.L.ref_ba_bookkeeping.restype = C.c_int
    n = r.L.ref_ba_bookkeeping(r.o, drop_target, remove_every, out, 20000)
    assert 0 < n <= 20000
    got["dropin"] = np.array(out[:n])
    assert np.array_equal(got["ref"], got["dropin"])
    nF, nP_counter, nR, nAll = got["ref"][:4]
    assert nF == win.nF and nAll == win.nP - (0 if remove_every <= 0 else len(range(0, win.nP, remove_every)))
    assert nR > 0 and (drop_target >= 0 or remove_every > 0 or nR == win.nR)


@needs_dropin
@pytest.mark.parametrize("geom", make_golden.MAKE_K_GEOMETRIES)
def test_dropin_tracker_make_k_matches_reference(geom):
    """CoarseTracker(w, h) + makeK of the drop-in unit (ldso_b200/host/dropin/dropin_tracker.cc) against the reference's CoarseTracker.cc
    (stored in tests/golden/reference_small.npz): the public per-level w, h, fx, fy, cx, cy and inverse intrinsics, bit for bit. Host
    logic only (the drop-in's device context cannot be created here and says so on stderr; makeK's host side does not depend on it)."""
    import ctypes as C
    w, h, levels, K = geom
    K = np.array(K, np.float64)
    got = {"ref": oracle_py.reference_golden()[f"make_k_{w}x{h}"]}
    L = oracle_py.ref_lib(oracle_py.DROPIN_LIB)
    out = np.zeros(10 * levels)
    L.ref_tracker_make_k.restype = C.c_int
    assert L.ref_tracker_make_k(w, h, levels, K.ctypes.data_as(C.POINTER(C.c_double)), out.ctypes.data_as(C.POINTER(C.c_double))) == levels
    got["dropin"] = out
    assert np.array_equal(got["ref"], got["dropin"])
    assert got["ref"][0] == w and got["ref"][10 * (levels - 1)] == w >> (levels - 1)


def test_select_activation_golden():
    """The frozen selection case (tests/golden/select_small.npz, written by tests/golden/make_golden.py from the pinned oracle)."""
    win, newest, args, flagged = make_golden.select_case()
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "select_small.npz"))
    o = oracle_py.OracleBA(win, threads_mode=0)
    for key, dist in (("13", 1.3), ("20", 2.0)):
        act, dmap = o.select_activation(newest, dist, *args, frame_flagged=flagged)
        assert np.array_equal(act, g["action" + key]) and np.array_equal(dmap.astype(np.uint16), g["map" + key])
    _, m0 = o.select_activation(newest, 2.0, *(a[:0] for a in args), frame_flagged=flagged)
    assert np.array_equal(m0.astype(np.uint16), g["map_seed_only"])


def test_reference_tracker_matches_oracle():
    """The reference's own CoarseTracker::trackNewestCoarse (optimised build in libref_ba.so, result stored in
    tests/golden/reference_small.npz) and the oracle port find the same pose and brightness on the full-size pair (the bit-exact
    comparison of the IEEE builds is oracle/ref_pin's)."""
    g = oracle_py.reference_golden()
    pair = make_golden.ref_track_pair("full")
    r = (bool(g["track_full_ok"]), g["track_full_R"], g["track_full_t"], *g["track_full_aff"])
    o = oracle_py.OracleTracker(pair, fast=True).track(np.eye(3), np.zeros(3), 0.0, 0.0, pair.levels - 1)
    assert r[0] and o[0]
    assert np.abs(r[2] - o[2]).max() < 1e-5 and np.abs(r[1] - o[1]).max() < 1e-5 and abs(r[3] - o[3]) < 1e-4 and abs(r[4] - o[4]) < 1e-2
    assert np.linalg.norm(r[2] - pair.t_true) < 0.05 * np.linalg.norm(pair.t_true)
