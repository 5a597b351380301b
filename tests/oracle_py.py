"""ctypes driver for the CPU oracle (oracle/liboracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs. The product package (ldso_b200/) never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")

_libs = {}

c_fp = C.POINTER(C.c_float)
c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int)
c_bp = C.POINTER(C.c_ubyte)


def build(force=False):
    need = force or not all(os.path.exists(os.path.join(ORACLE_DIR, n)) for n in ("liboracle.so", "liboracle_fast.so"))
    if not need:
        srcs = [os.path.join(ORACLE_DIR, f) for f in os.listdir(ORACLE_DIR) if f.endswith((".cc", ".h"))]
        newest = max(os.path.getmtime(s) for s in srcs)
        need = newest > os.path.getmtime(os.path.join(ORACLE_DIR, "liboracle.so"))
    if need:
        subprocess.check_call(["make", "-C", ORACLE_DIR, "-s"])


def lib(fast=False):
    key = "fast" if fast else "ieee"
    if key not in _libs:
        build()
        L = C.CDLL(os.path.join(ORACLE_DIR, "liboracle_fast.so" if fast else "liboracle.so"))
        L.oracle_ba_create.restype = C.c_void_p
        L.oracle_ba_create.argtypes = [C.c_int, C.c_int, C.c_int]
        L.oracle_ba_destroy.argtypes = [C.c_void_p]
        L.oracle_ba_optimize_begin.restype = C.c_double
        L.oracle_ba_linearize_all.restype = C.c_double
        L.oracle_ba_last_energy.restype = C.c_double
        L.oracle_ba_calc_m_energy.restype = C.c_double
        L.oracle_ba_calc_l_energy.restype = C.c_double
        L.oracle_ba_time_gn.restype = C.c_double
        L.oracle_tracker_create.restype = C.c_void_p
        _libs[key] = L
    return _libs[key]


def _f(a):
    return a.ctypes.data_as(c_fp)


def _d(a):
    return a.ctypes.data_as(c_dp)


REF_LIB = os.path.join(ORACLE_DIR, "_ref", "libref_ba.so")


DROPIN_LIB = os.path.join(ORACLE_DIR, "_ref", "libdropin_ba.so")


def reference_golden():
    """What the reference's own translation units (libref_ba.so) computed on the cases of the tests that compare with the reference:
    tests/golden/reference_small.npz, written by `python tests/golden/make_golden.py --reference`."""
    return np.load(os.path.join(ROOT, "tests", "golden", "reference_small.npz"))


def ref_lib(path=None):
    """oracle/_ref/libref_ba.so: the reference's own back-end translation units behind a C interface (oracle/ref_pin/ref_bench.cc).
    Built by `make -C oracle ref_pin` where /root/reference is mounted; None where it is not there (the built file travels).
    path = DROPIN_LIB: the same interface and driver over the product's drop-in translation units (ldso_b200/host/dropin/*.cc:
    the reference's class declarations, forwarding to libldso_b200.so) instead of the reference's own five."""
    path = path or REF_LIB
    if not os.path.exists(path):
        return None
    L = C.CDLL(path)
    L.ref_ba_create.restype = C.c_void_p
    for f in ("ref_ba_optimize_begin", "ref_ba_energy", "ref_ba_time_gn"):
        getattr(L, f).restype = C.c_double
    return L


class RefBA:
    """The same window as OracleBA, held by the REFERENCE'S own classes (FrameHessian, PointHessian, PointFrameResidual,
    EnergyFunctional, IndexThreadReduce) compiled from /root/reference; only FullSystem.cc's driver loop is restated around them."""

    def __init__(self, win, multithreaded=True, calib_delta=None, lib_path=None):
        self.L = ref_lib(lib_path)
        if self.L is None:
            raise RuntimeError("oracle/_ref/libref_ba.so is not built (needs the reference tree: make -C oracle ref_pin)")
        self.win = win
        self.o = C.c_void_p(self.L.ref_ba_create(win.w, win.h, int(bool(multithreaded))))
        self._keep = []
        K = np.ascontiguousarray(win.K, np.float64)
        cd = None if calib_delta is None else np.ascontiguousarray(calib_delta, np.float64)
        self.L.ref_ba_set_calib(self.o, _d(K), None if cd is None else _d(cd))
        for i in range(win.nF):
            dI = np.ascontiguousarray(win.pyramids[i][0], np.float32)
            self._keep.append(dI)
            self.L.ref_ba_add_frame(self.o, _d(np.ascontiguousarray(win.Rcw[i], np.float64)), _d(np.ascontiguousarray(win.tcw[i], np.float64)),
                                    _d(np.ascontiguousarray(win.state_zero[i], np.float64)), _d(np.ascontiguousarray(win.state[i], np.float64)),
                                    C.c_float(float(win.ab_exposure[i])), int(win.frame_id[i]), _f(dI))
        col = np.ascontiguousarray(win.pt_color, np.float32)
        wts = np.ascontiguousarray(win.pt_weights, np.float32)
        for p in range(win.nP):
            self.L.ref_ba_add_point(self.o, int(win.pt_host[p]), C.c_float(float(win.pt_u[p])), C.c_float(float(win.pt_v[p])),
                                    C.c_float(float(win.pt_idepth_zero[p])), C.c_float(float(win.pt_idepth[p])), int(win.pt_has_prior[p]),
                                    _f(col[p]), _f(wts[p]))
        for r in range(win.nR):
            self.L.ref_ba_add_residual(self.o, int(win.res_point[r]), int(win.res_target[r]))
        self.L.ref_ba_finalize(self.o)
        self.n = 8 * win.nF + 4

    def optimize_begin(self):
        return self.L.ref_ba_optimize_begin(self.o)

    def gn_iteration(self, it):
        return bool(self.L.ref_ba_gn_iteration(self.o, it))

    def energy(self):
        return self.L.ref_ba_energy(self.o)

    def time_gn(self, iters, warmup):
        return self.L.ref_ba_time_gn(self.o, iters, warmup)

    def last_x(self):
        x = np.zeros(self.n, np.float64)
        self.L.ref_ba_last_x(self.o, _d(x))
        return x

    def idepths(self):
        a = np.zeros(self.win.nP, np.float32)
        self.L.ref_ba_point_idepths(self.o, _f(a))
        return a


class RefTracker:
    """The reference's own CoarseTracker (src/frontend/CoarseTracker.cc in oracle/_ref/libref_ba.so) on a synth.make_track_pair() case."""

    def __init__(self, pair, lib_path=None):
        self.L = ref_lib(lib_path)
        if self.L is None:
            raise RuntimeError("oracle/_ref/libref_ba.so is not built")
        self.L.ref_tracker_create.restype = C.c_void_p
        self.pair = pair
        self._ref = [np.ascontiguousarray(p, np.float32) for p in pair.ref_pyr]
        self._new = [np.ascontiguousarray(p, np.float32) for p in pair.new_pyr]
        ref_arr = (c_fp * pair.levels)(*[_f(p) for p in self._ref])
        new_arr = (c_fp * pair.levels)(*[_f(p) for p in self._new])
        cpt = np.ascontiguousarray(pair.cpt, np.float32)
        hd = np.ascontiguousarray(pair.HdiF, np.float32)
        K = np.ascontiguousarray(pair.K, np.float64)
        self.o = C.c_void_p(self.L.ref_tracker_create(pair.w, pair.h, pair.levels, _d(K), ref_arr, C.c_float(pair.ref_aff[0]), C.c_float(pair.ref_aff[1]),
                                                      C.c_float(1.0), len(hd), _f(cpt), _f(hd), new_arr, C.c_float(1.0)))

    def track(self, R, t, aff_a, aff_b, coarsest, reps=1):
        """(ok, R, t, a, b, seconds per call)"""
        R = np.ascontiguousarray(R, np.float64).copy()
        t = np.ascontiguousarray(t, np.float64).copy()
        a, b, sec = C.c_float(aff_a), C.c_float(aff_b), C.c_double(0.0)
        ok = self.L.ref_tracker_track(self.o, _d(R), _d(t), C.byref(a), C.byref(b), int(coarsest), int(reps), C.byref(sec))
        return bool(ok), R, t, a.value, b.value, sec.value


class OracleBA:
    """One oracle window built from a ldso_b200.synth.Window."""

    def __init__(self, win, threads_mode=0, fast=False, calib_delta=None):
        self.L = lib(fast)
        self.win = win
        self.o = C.c_void_p(self.L.oracle_ba_create(win.w, win.h, threads_mode))
        self._keep = []
        K = np.ascontiguousarray(win.K, np.float64)
        self.L.oracle_ba_set_calib(self.o, _d(K))
        if calib_delta is not None:
            cd = np.ascontiguousarray(calib_delta, np.float64)
            self.L.oracle_ba_set_calib_delta(self.o, _d(cd))
        for i in range(win.nF):
            dI = np.ascontiguousarray(win.pyramids[i][0], np.float32)
            self._keep.append(dI)
            R = np.ascontiguousarray(win.Rcw[i], np.float64)
            t = np.ascontiguousarray(win.tcw[i], np.float64)
            sz = np.ascontiguousarray(win.state_zero[i], np.float64)
            st = np.ascontiguousarray(win.state[i], np.float64)
            self.L.oracle_ba_add_frame(self.o, _d(R), _d(t), _d(sz), _d(st), C.c_float(float(win.ab_exposure[i])),
                                       int(win.frame_id[i]), _f(dI))
        col = np.ascontiguousarray(win.pt_color, np.float32)
        wts = np.ascontiguousarray(win.pt_weights, np.float32)
        for p in range(win.nP):
            self.L.oracle_ba_add_point(self.o, int(win.pt_host[p]), C.c_float(float(win.pt_u[p])), C.c_float(float(win.pt_v[p])),
                                       C.c_float(float(win.pt_idepth_zero[p])), C.c_float(float(win.pt_idepth[p])),
                                       int(win.pt_has_prior[p]), _f(col[p]), _f(wts[p]))
        rp = win.res_point
        for r in range(win.nR):
            self.L.oracle_ba_add_residual(self.o, int(rp[r]), int(win.res_target[r]))
        self.L.oracle_ba_finalize(self.o)
        self.n = 8 * win.nF + 4

    def __del__(self):
        try:
            self.L.oracle_ba_destroy(self.o)
        except Exception:
            pass

    def set_marg_prior(self, HM, bM):
        HMc = np.asfortranarray(HM, np.float64)
        bMc = np.ascontiguousarray(bM, np.float64)
        self.L.oracle_ba_set_marg_prior(self.o, HMc.ctypes.data_as(c_dp), _d(bMc))

    def optimize_begin(self):
        return self.L.oracle_ba_optimize_begin(self.o)

    def gn_iteration(self, it):
        return bool(self.L.oracle_ba_gn_iteration(self.o, it))

    def energy(self):
        """lastEnergyP of the last linearizeAll."""
        return self.L.oracle_ba_last_energy(self.o)

    def calc_energies(self):
        """(calcLEnergyF_MT, calcMEnergyF) at the current state."""
        return self.L.oracle_ba_calc_l_energy(self.o), self.L.oracle_ba_calc_m_energy(self.o)

    def linearize_all(self, fix=False):
        return self.L.oracle_ba_linearize_all(self.o, int(fix))

    def apply_res(self):
        self.L.oracle_ba_apply_res(self.o)

    def solve_system(self, it):
        self.L.oracle_ba_solve_system(self.o, it)

    def do_step(self):
        return bool(self.L.oracle_ba_do_step(self.o))

    def time_gn(self, iters, warmup):
        return self.L.oracle_ba_time_gn(self.o, iters, warmup)

    def system(self):
        n = self.n
        mats = {k: np.zeros((n, n), np.float64, order="F") for k in ("HA", "Hsc", "lastHS", "HL")}
        vecs = {k: np.zeros(n, np.float64) for k in ("bA", "bsc", "lastbS", "lastX", "bL")}
        self.L.oracle_ba_get_system(self.o, _d(mats["HA"]), _d(vecs["bA"]), _d(mats["Hsc"]), _d(vecs["bsc"]),
                                    _d(mats["lastHS"]), _d(vecs["lastbS"]), _d(vecs["lastX"]), _d(mats["HL"]), _d(vecs["bL"]))
        out = dict(mats)
        out.update(vecs)
        return out

    def marg_prior(self, n=None):
        n = self.n if n is None else n
        HM = np.zeros((n, n), np.float64, order="F")
        bM = np.zeros(n, np.float64)
        self.L.oracle_ba_get_marg_prior(self.o, _d(HM), _d(bM))
        return HM, bM

    def optimize_immature(self, u, v, host, idepth_min, idepth_max, color, weights, energyTH, min_obs=1):
        """FullSystem::optimizeImmaturePoint for every candidate against the window's current frame states."""
        n = len(u)
        f32 = lambda a: np.ascontiguousarray(a, np.float32)
        u, v, imin, imax, col, wts, eth = map(f32, (u, v, idepth_min, idepth_max, color, weights, energyTH))
        host = np.ascontiguousarray(host, np.int32)
        ok = np.zeros(n, np.int32); idepth = np.zeros(n, np.float32); states = np.zeros((n, self.win.nF), np.uint8)
        self.L.oracle_ba_optimize_immature(self.o, n, _f(u), _f(v), host.ctypes.data_as(c_ip), _f(imin), _f(imax), _f(col), _f(wts), _f(eth),
                                           int(min_obs), ok.ctypes.data_as(c_ip), _f(idepth), states.ctypes.data_as(C.POINTER(C.c_ubyte)))
        return ok, idepth, states

    def select_activation(self, newest, current_min_act_dist, u, v, host, idepth_min, idepth_max, status, interval, quality, my_type,
                          frame_flagged=None, min_trace_quality=3.0, levels=None):
        """FullSystem::activatePointsMT's selection loop (CoarseDistanceMap + the greedy pass): (action[n], dist_map[h/2, w/2])."""
        f32 = lambda a: np.ascontiguousarray(a, np.float32)
        u, v, imin, imax, itv, q, mt = map(f32, (u, v, idepth_min, idepth_max, interval, quality, my_type))
        host = np.ascontiguousarray(host, np.int32); status = np.ascontiguousarray(status, np.int32)
        n = u.shape[0]
        flagged = np.zeros(self.win.nF, np.uint8) if frame_flagged is None else np.ascontiguousarray(frame_flagged, np.uint8)
        action = np.zeros(n, np.uint8)
        dmap = np.zeros((self.win.h >> 1, self.win.w >> 1), np.float32)
        ub = C.POINTER(C.c_ubyte)
        self.L.oracle_ba_select_activation(self.o, int(levels or self.win.levels), int(newest), C.c_float(current_min_act_dist), C.c_float(min_trace_quality), n,
                                           _f(u), _f(v), host.ctypes.data_as(c_ip), _f(imin), _f(imax), status.ctypes.data_as(c_ip), _f(itv), _f(q), _f(mt),
                                           flagged.ctypes.data_as(ub), action.ctypes.data_as(ub), _f(dmap))
        return action, dmap

    def marginalize_frame(self, idx):
        """EnergyFunctional::marginalizeFrame's HM/bM algebra; returns the shrunken (HM, bM)."""
        nd = int(self.L.oracle_ba_marginalize_frame(self.o, int(idx)))
        return self.marg_prior(nd)

    def res_counts(self):
        a, l, m = C.c_int(), C.c_int(), C.c_int()
        self.L.oracle_ba_res_counts(self.o, C.byref(a), C.byref(l), C.byref(m))
        return a.value, l.value, m.value

    def points(self):
        nP = self.win.nP
        keys = ("idepth", "idepth_zero", "step", "HdiF", "bdSumF", "Hdd_accAF", "bd_accAF")
        out = {k: np.zeros(nP, np.float32) for k in keys}
        out["Hcd_accAF"] = np.zeros((nP, 4), np.float32)
        out["deltaF"] = np.zeros(nP, np.float32)
        self.L.oracle_ba_get_points(self.o, *[_f(out[k]) for k in keys], _f(out["Hcd_accAF"]), _f(out["deltaF"]))
        return out

    def residuals(self):
        nR = self.win.nR
        out = dict(
            state_state=np.zeros(nR, np.int32), state_NewState=np.zeros(nR, np.int32),
            state_energy=np.zeros(nR, np.float64), state_NewEnergy=np.zeros(nR, np.float64),
            state_NewEnergyWithOutlier=np.zeros(nR, np.float64), J=np.zeros((nR, 74), np.float32),
            JpJdF=np.zeros((nR, 8), np.float32), projectedTo=np.zeros((nR, 8, 2), np.float32),
            centerProjectedTo=np.zeros((nR, 3), np.float32), isActive=np.zeros(nR, np.uint8),
            isLinearized=np.zeros(nR, np.uint8), res_toZeroF=np.zeros((nR, 8), np.float32))
        self.L.oracle_ba_get_residuals(
            self.o, out["state_state"].ctypes.data_as(c_ip), out["state_NewState"].ctypes.data_as(c_ip),
            _d(out["state_energy"]), _d(out["state_NewEnergy"]), _d(out["state_NewEnergyWithOutlier"]), _f(out["J"]),
            _f(out["JpJdF"]), _f(out["projectedTo"]), _f(out["centerProjectedTo"]),
            out["isActive"].ctypes.data_as(c_bp), out["isLinearized"].ctypes.data_as(c_bp), _f(out["res_toZeroF"]))
        return out

    def frames(self):
        nF = self.win.nF
        out = dict(state=np.zeros((nF, 10)), step=np.zeros((nF, 10)), frameEnergyTH=np.zeros(nF, np.float32),
                   precalc=np.zeros((nF * nF, 40), np.float32), adHost=np.zeros((nF * nF, 8, 8)),
                   adTarget=np.zeros((nF * nF, 8, 8)), adHTdeltaF=np.zeros((nF * nF, 8), np.float32),
                   calib_value=np.zeros(4), prior=np.zeros((nF, 8)), delta_prior=np.zeros((nF, 8)), delta=np.zeros((nF, 8)))
        self.L.oracle_ba_get_frames(self.o, _d(out["state"]), _d(out["step"]), _f(out["frameEnergyTH"]), _f(out["precalc"]),
                                    _d(out["adHost"]), _d(out["adTarget"]), _f(out["adHTdeltaF"]), _d(out["calib_value"]),
                                    _d(out["prior"]), _d(out["delta_prior"]), _d(out["delta"]))
        return out

    def nullspace_projector(self):
        n = self.n
        P = np.zeros((n, n), np.float64, order="F")
        self.L.oracle_ba_get_nullspace_projector(self.o, _d(P))
        return P

    def marginalize_points(self, idx, prior_fac=600.0 * 600.0):
        idx = np.ascontiguousarray(idx, np.int32)
        self.L.oracle_ba_marginalize_points(self.o, len(idx), idx.ctypes.data_as(c_ip), C.c_float(prior_fac))


def make_images(color, levels, fast=False):
    L = lib(fast)
    h, w = color.shape
    color = np.ascontiguousarray(color, np.float32)
    outs = [np.zeros(((h >> l), (w >> l), 3), np.float32) for l in range(levels)]
    arr = (c_fp * levels)(*[_f(o) for o in outs])
    L.oracle_make_images(_f(color), w, h, levels, arr)
    return outs


class OracleTracker:
    def __init__(self, pair, fast=False):
        self.L = lib(fast)
        self.pair = pair
        self.levels = pair.levels
        self.o = C.c_void_p(self.L.oracle_tracker_create(pair.w, pair.h, pair.levels))
        K = pair.K
        self.L.oracle_tracker_make_k(self.o, C.c_float(K[0]), C.c_float(K[1]), C.c_float(K[2]), C.c_float(K[3]))
        self._ref = [np.ascontiguousarray(p, np.float32) for p in pair.ref_pyr]
        self._new = [np.ascontiguousarray(p, np.float32) for p in pair.new_pyr]
        ref_arr = (c_fp * self.levels)(*[_f(p) for p in self._ref])
        new_arr = (c_fp * self.levels)(*[_f(p) for p in self._new])
        cpt = np.ascontiguousarray(pair.cpt, np.float32)
        hd = np.ascontiguousarray(pair.HdiF, np.float32)
        self.L.oracle_tracker_set_ref(self.o, ref_arr, C.c_float(pair.ref_aff[0]), C.c_float(pair.ref_aff[1]),
                                      C.c_float(1.0), len(hd), _f(cpt), _f(hd))
        self.L.oracle_tracker_set_new_frame(self.o, new_arr, C.c_float(1.0))

    def __del__(self):
        try:
            self.L.oracle_tracker_destroy(self.o)
        except Exception:
            pass

    def pc(self, lvl):
        n = self.L.oracle_tracker_pc_n(self.o, lvl)
        a = [np.zeros(n, np.float32) for _ in range(4)]
        self.L.oracle_tracker_get_pc(self.o, lvl, *[_f(x) for x in a])
        return a

    def eval(self, lvl, R, t, aff_a, aff_b, cutoff, with_H=True):
        R = np.ascontiguousarray(R, np.float64)
        t = np.ascontiguousarray(t, np.float64)
        res = np.zeros(6)
        H = np.zeros((8, 8))
        b = np.zeros(8)
        self.L.oracle_tracker_eval(self.o, lvl, _d(R), _d(t), C.c_float(aff_a), C.c_float(aff_b), C.c_float(cutoff),
                                   _d(res), _d(H) if with_H else None, _d(b) if with_H else None)
        return res, H, b

    def track(self, R, t, aff_a, aff_b, coarsest, min_res=None):
        R = np.array(R, np.float64, order="C")
        t = np.array(t, np.float64)
        a = C.c_float(aff_a)
        b = C.c_float(aff_b)
        mr = np.full(5, np.nan) if min_res is None else np.ascontiguousarray(min_res, np.float64)
        lr = np.zeros(5)
        lf = np.zeros(3)
        ne = C.c_int()
        ok = self.L.oracle_tracker_track(self.o, _d(R), _d(t), C.byref(a), C.byref(b), coarsest, _d(mr), _d(lr), _d(lf),
                                         C.byref(ne))
        return bool(ok), R, t, a.value, b.value, lr, lf, ne.value


# ---- immature-point trace (oracle/trace.cc) -------------------------------------------------------------
IPS_GOOD, IPS_OOB, IPS_OUTLIER, IPS_SKIPPED, IPS_BADCONDITION, IPS_UNINITIALIZED = range(6)


class OracleTrace:
    """ImmaturePoint candidates of a synth.TraceCase and FullSystem::traceNewCoarse passes over them."""

    def __init__(self, win, case):
        self.L = lib()
        self.win, self.case = win, case
        n = case.n
        self.color = np.zeros((n, 8), np.float32); self.weights = np.zeros((n, 8), np.float32)
        self.gradH = np.zeros((n, 4), np.float32); self.energyTH = np.zeros(n, np.float32)
        for h in np.unique(case.host):
            m = np.nonzero(case.host == h)[0]
            dI = np.ascontiguousarray(win.pyramids[h][0], np.float32)
            u = np.ascontiguousarray(case.u[m]); v = np.ascontiguousarray(case.v[m])
            c = np.zeros((len(m), 8), np.float32); wt = np.zeros((len(m), 8), np.float32); g = np.zeros((len(m), 4), np.float32)
            e = np.zeros(len(m), np.float32)
            self.L.oracle_trace_init(_f(dI), win.w, len(m), _f(u), _f(v), _f(c), _f(wt), _f(g), _f(e))
            self.color[m], self.weights[m], self.gradH[m], self.energyTH[m] = c, wt, g, e
        self.idepth_min = np.zeros(n, np.float32); self.idepth_max = np.full(n, np.nan, np.float32)
        self.quality = np.full(n, 10000.0, np.float32); self.status = np.full(n, IPS_UNINITIALIZED, np.int32)
        self.uv = np.zeros((n, 2), np.float32); self.interval = np.zeros(n, np.float32)

    def trace_on(self, new):
        c, win = self.case, self.win
        dI = np.ascontiguousarray(win.pyramids[new][0], np.float32)
        KRKi = np.ascontiguousarray(c.KRKi[new]); Kt = np.ascontiguousarray(c.Kt[new]); aff = np.ascontiguousarray(c.aff[new])
        self.L.oracle_trace_on(_f(dI), win.w, win.h, c.n, _f(c.u), _f(c.v), _f(self.color), _f(self.weights), _f(self.gradH),
                               _f(self.energyTH), c.host.ctypes.data_as(c_ip), _f(KRKi), _f(Kt), _f(aff), _f(self.idepth_min),
                               _f(self.idepth_max), _f(self.quality), self.status.ctypes.data_as(c_ip), _f(self.uv), _f(self.interval))
        return self.status.copy()


def se3_log(R, t, fast=False):
    """Sophus SE3::log of (R, t): (upsilon[3], omega[3])."""
    L = lib(fast)
    R = np.ascontiguousarray(R, np.float64); t = np.ascontiguousarray(t, np.float64)
    a = np.zeros(6, np.float64)
    L.oracle_se3_log(_d(R), _d(t), _d(a))
    return a


def init_calc_res(pair, lvl, R, t, aff_a, aff_b, u, v, idepth_new, iR, isGood, energy2, outlierTH, alphaK=2.5 * 2.5, alphaW=150.0 * 150.0,
                  couplingWeight=1.0, fast=False):
    """CoarseInitializer::calcResAndGS (oracle/initializer.cc) on the pyramids of a synth.make_track_pair() case: first frame = ref, new = new."""
    L = lib(fast)
    ref = [np.ascontiguousarray(p, np.float32) for p in pair.ref_pyr]
    new = [np.ascontiguousarray(p, np.float32) for p in pair.new_pyr]
    ra = (c_fp * pair.levels)(*[_f(p) for p in ref]); na = (c_fp * pair.levels)(*[_f(p) for p in new])
    f32 = lambda a: np.ascontiguousarray(a, np.float32)
    u, v, idn, iR, e2, oth = map(f32, (u, v, idepth_new, iR, energy2, outlierTH))
    good = np.ascontiguousarray(isGood, np.uint8)
    n = u.shape[0]
    K = np.ascontiguousarray(pair.K, np.float64); R = np.ascontiguousarray(R, np.float64); t = np.ascontiguousarray(t, np.float64)
    out = dict(isGood_new=np.zeros(n, np.uint8), energy_new=np.zeros((n, 2), np.float32), maxstep=np.zeros(n, np.float32),
               lastHessian_new=np.zeros(n, np.float32), Jb=np.zeros((n, 10), np.float32), H=np.zeros((8, 8), np.float32), b=np.zeros(8, np.float32),
               Hsc=np.zeros((8, 8), np.float32), bsc=np.zeros(8, np.float32), res=np.zeros(3, np.float32))
    ub = C.POINTER(C.c_ubyte)
    L.oracle_init_calc_res(pair.w, pair.h, pair.levels, _d(K), ra, na, int(lvl), _d(R), _d(t), C.c_float(aff_a), C.c_float(aff_b), n, _f(u), _f(v), _f(idn),
                           _f(iR), good.ctypes.data_as(ub), _f(e2), _f(oth), C.c_float(alphaK), C.c_float(alphaW), C.c_float(couplingWeight),
                           out["isGood_new"].ctypes.data_as(ub), _f(out["energy_new"]), _f(out["maxstep"]), _f(out["lastHessian_new"]), _f(out["Jb"]),
                           _f(out["H"]), _f(out["b"]), _f(out["Hsc"]), _f(out["bsc"]), _f(out["res"]))
    return out
