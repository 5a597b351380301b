#!/usr/bin/env python
"""bench.py — GN-iterations/sec of the photometric BA hot path (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps K --warmup W            # our CUDA arm (N=1: 8 KF x 2000 active points)
    torchrun ... bench.py --gpus N ...                        # points sharded over N ranks, one NCCL all-reduce/step
    python bench.py --impl reference ...                      # the reference's CPU path (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's outputs as DIR/<name>.npy

One "step" = one Gauss-Newton iteration (FullSystem.cc:777-831 restricted to the path): accumulate + Schur +
stitch + 68x68 solve + resubstitute + state step + 64 frame-pair precalcs + linearize all residuals + applyRes.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "GN-iters/sec, 8-KF x 2k-point window; Hessian rel-err vs SSE ref"
PTS_PER_FRAME = 250       # per GPU: 8 KF x 250 = 2000 active points (BASELINE.json configs[1])
NF = 8
E2E_CONTEXTS = 4          # windows in flight in the end-to-end leg (one host thread, one stream per context)


def common_config(n_gpus, n_points, n_residuals):
    """The workload description both arms print verbatim (the driver compares the two `config` objects)."""
    return {"workload": f"8 KF x {PTS_PER_FRAME * NF} active points per GPU: one 8 KF x {n_points}-point sliding window "
                        f"({n_residuals} residuals), 640x480, seed 42; value counts {n_gpus} x (window iterations / s), i.e. 2000-point-window iterations / s",
            "nF": NF, "n_gpus": n_gpus, "n_points": int(n_points), "n_residuals": int(n_residuals), "points_per_gpu": PTS_PER_FRAME * NF}


def algorithmic_bytes(n_res, n_pts, nF):
    """SURVEY.md §8d: bytes the reference's algorithm must touch once per GN iteration."""
    n = 8 * nF + 4
    return n_res * (384 + 12 + 12) + n_pts * (80 + 8 + 4) + nF * nF * 1164 + 4 * (n * n + n) * 8


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe). The timed region of this bench is
    milliseconds long (20 steps x ~60 us), far below nvidia-smi's 100 ms period, so the samples are taken through NVML itself: one
    sample right before the loop, a polling thread (~2 kHz) while it runs, one right after. Falls back to one nvidia-smi query
    before/after when NVML cannot be loaded."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.stop_flag = False
        self.h = None
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        except Exception:  # noqa: BLE001
            self.nv = None

    def _one(self):
        if self.nv is not None:
            nv = self.nv
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((float(sm), float(mx), int(rs)))
            except Exception:  # noqa: BLE001
                pass
        else:
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active"
            try:
                r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.gpu)],
                                   capture_output=True, text=True, timeout=5)
                f = [x.strip() for x in r.stdout.strip().split(",")]
                self.rows.append((float(f[0]), float(f[1]), int(f[2], 16)))
            except Exception:  # noqa: BLE001
                pass

    def _poll(self):
        while not self.stop_flag:
            self._one()
            time.sleep(0.0005)

    def start(self):
        self._one()
        self.th = None
        if self.nv is not None:
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.th is not None:
            self.th.join(timeout=2)
        self._one()
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["no clock source (NVML and nvidia-smi unavailable)"]}
        sm = [r[0] for r in self.rows]
        reasons = set()
        for r in self.rows:
            for bit, nm in self.REASONS.items():
                if r[2] & bit:
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)), "sm_mhz_min": float(min(sm)), "sm_max_mhz": float(max(r[1] for r in self.rows)),
                "samples": len(sm), "reasons": sorted(reasons), "source": "NVML polled before / during / after the timed loop" if self.nv else "nvidia-smi before / after"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------------------------- reference arm
def _ref_arm_seconds_per_iter(steps, warmup, pts_per_frame=PTS_PER_FRAME):
    """Seconds per GN iteration of the REFERENCE'S OWN back end (oracle/_ref/libref_ba.so: the reference's translation units compiled
    unmodified against stand-in Eigen headers, its own 6-thread IndexThreadReduce; oracle/ref_pin/ref_bench.cc) on the bench window, or
    None when that library is not there or does not run on this host. A child process: a library built with -march=native elsewhere
    must not be able to take the bench down."""
    here = os.path.dirname(os.path.abspath(__file__))
    if not os.path.exists(os.path.join(here, "oracle", "_ref", "libref_ba.so")):
        return None
    code = ("import time\nfrom ldso_b200 import synth\nfrom tests import oracle_py\n"
            f"win = synth.make_window(nF={NF}, pts_per_frame={int(pts_per_frame)}, seed=42)\n"
            "r = oracle_py.RefBA(win, multithreaded=True)\nr.optimize_begin()\n"
            f"[r.gn_iteration(min(i, 3)) for i in range({int(warmup)})]\n"
            f"t0 = time.perf_counter()\n[r.gn_iteration(3) for _ in range({int(steps)})]\n"
            f"print('REFARM', (time.perf_counter() - t0) / {int(steps)})\n")
    import subprocess
    try:
        r = subprocess.run([sys.executable, "-c", code], cwd=here, capture_output=True, text=True, timeout=900)
    except Exception:
        return None
    for ln in r.stdout.splitlines():
        if ln.startswith("REFARM "):
            return float(ln.split()[1])
    return None


def _port_seconds_per_iter(win, steps, warmup):
    from tests import oracle_py
    o = oracle_py.OracleBA(win, threads_mode=6, fast=True)
    o.optimize_begin()
    for i in range(warmup):
        o.gn_iteration(min(i, 3))
    t0 = time.perf_counter()
    for i in range(steps):
        o.gn_iteration(3)
    return (time.perf_counter() - t0) / steps


def run_reference(args):
    """The reference's own CPU implementation of the path, on the host cores, with the reference's hard-wired 6 worker threads
    (NUM_THREADS, include/Settings.h:9). LDSO's build cannot run here (Eigen / glog / OpenCV / Pangolin absent), but its back-end
    translation units compile unmodified against stand-in Eigen headers: oracle/_ref/libref_ba.so (kind "reference": linearize, both
    addPoint's, the stitchers, solveSystemF, resubstituteF and IndexThreadReduce are the reference's code; FullSystem.cc's driver loop
    around them is restated in oracle/ref_pin/ref_bench.cc; the 68x68 dense algebra runs through the stand-in). When that library is not
    there, the oracle port (oracle/liboracle_fast.so, kind "port"). The port's rate is reported beside it either way."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from ldso_b200 import synth
    # the same window the GPU arm iterates at this N (weak scaling: 2000 points per GPU -> 2000*N points here, on the host CPU)
    world = max(1, args.gpus)
    win = synth.make_window(nF=NF, pts_per_frame=PTS_PER_FRAME * world, seed=42)
    sec_port = _port_seconds_per_iter(win, args.steps, args.warmup)
    sec_ref = _ref_arm_seconds_per_iter(args.steps, args.warmup, PTS_PER_FRAME * world)
    kind = "reference" if sec_ref else "port"
    sec = sec_ref if sec_ref else sec_port
    v = world / sec            # 2000-point-window iterations per second, the unit of the GPU arm's value
    cores = os.cpu_count()
    what = ("the reference's own Residuals.cc / AccumulatedTopHessian.cc / AccumulatedSCHessian.cc / EnergyFunctional.cc / FrameHessian.cc / "
            "FrameFramePrecalc.cc compiled -O3 -march=native against stand-in Eigen headers (oracle/_ref/libref_ba.so), its own IndexThreadReduce"
            if sec_ref else "oracle port (g++ -O3 -march=native)")
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "GN-iters/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": common_config(world, win.nP, win.nR),
        "window_iters_per_s": 1.0 / sec,
        "cpu_baseline": {"value": v, "unit": "GN-iters/s", "cores": 6, "kind": kind, "port_value": world / sec_port,
                         "sample": f"{args.steps} full GN iterations of the same {win.nP}-point window; {what}, 6 worker threads "
                                   f"(reference NUM_THREADS) on a {cores}-core host; port_value = the oracle port on the same sample"},
        "e2e": {"value": v, "unit": "GN-iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------- our arm
class _DevBuf:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 3, "strides": None}


def run_ours(args):
    import torch
    from ldso_b200 import capi, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: ldso_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist  # noqa: F811
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node == --gpus"

    # weak scaling: 2000 points per GPU; the global window has 2000*N points, sharded by contiguous point blocks
    full = synth.make_window(nF=NF, pts_per_frame=PTS_PER_FRAME * world, seed=42)
    win = synth.shard_window(full, rank, world) if world > 1 else full
    stream = torch.cuda.Stream()          # a real (capturable) stream; everything below runs on it
    torch.cuda.set_stream(stream)
    ctx = capi.Context(win.w, win.h, win.levels, device=local_rank)
    ctx.set_stream(stream.cuda_stream)
    ctx.load_synth_window(win)
    red_t = None
    use_nccl = world > 1 and args.collective == "nccl"
    if world > 1:
        newest = full.nF - 1
        counts = []
        for r in range(world):
            w_r = synth.shard_window(full, r, world)
            counts.append(int(np.sum(w_r.res_target == newest)))
        ctx.set_shard(int(np.sum(counts[:rank])), int(np.sum(counts)))
        if use_nccl:
            ptr, n = ctx.reduce_buffer()
            red_t = torch.as_tensor(_DevBuf(ptr, n), device=f"cuda:{local_rank}")
        else:
            # device-side exchange: one kernel over NVLink peer memory per step (CUDA IPC handles travel through
            # torch.distributed once); the loop itself makes no NCCL call
            handles = [None] * world
            dist.all_gather_object(handles, ctx.peer_export())
            ctx.peer_connect(rank, world, handles)
            dist.barrier()

    def prologue():
        if use_nccl:
            ctx.gn_phase_a(-1)
            dist.all_reduce(red_t)
            ctx.gn_phase_b()
        else:
            ctx.optimize_begin(want_energy=False)

    def gn_step(it):
        if use_nccl:
            ctx.gn_phase_a(it)
            dist.all_reduce(red_t)
            ctx.gn_phase_b()
        else:
            ctx.gn_iterations(it, 1)

    flush = torch.empty(192 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    prologue()
    for i in range(max(args.warmup, 3)):
        gn_step(min(i, 3))
    torch.cuda.synchronize()
    launches0 = ctx.launch_count()

    # ---- timed region: K iterations, each bracketed by CUDA events on the launching stream, L2 flushed between
    sampler = ClockSampler(local_rank)
    sampler.start()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    wall0 = time.perf_counter()
    for k in range(args.steps):
        flush.fill_(k & 0xff)
        ev[k][0].record(stream)
        gn_step(3)
        ev[k][1].record(stream)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    wall = time.perf_counter() - wall0
    launches = ctx.launch_count() - launches0
    t_ms = float(sum(a.elapsed_time(b) for a, b in ev))
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(ctx, args.dump_outputs)

    # ---- same loop without the flush (images L2-resident, as inside a real optimize() call) — reported as extra
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()          # ranks leave the clock sampler at different times: start the loop together
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(args.steps):
        gn_step(3)
    e1.record(stream)
    torch.cuda.synchronize()
    t_warm_ms = e0.elapsed_time(e1)

    # ---- per-kernel durations (CUDA events around each launch, L2 flushed between iterations) for the roofline of the
    # dominant HBM kernel K1 (fused linearize + accumulate: it moves all of the per-residual / per-point algorithmic bytes)
    ctx.kernel_times(True)
    for k in range(min(args.steps, 50)):
        flush.fill_(k & 0xff)
        gn_step(3)
    ktimes = ctx.kernel_times(False)

    # ---- end-to-end through the C ABI with host buffers (single GPU arm only): every step uploads the newest
    # keyframe's raw image (device-side makeImages), the frame states and the whole window from host memory, runs
    # one GN iteration and reads the solution, energy, point idepths/steps and residual states back.
    e2e = None
    if world == 1:
        e2e = run_e2e(ctx, win, args, torch)

    trace_extra = None
    big_extra = None
    if world == 1:
        trace_extra = run_trace(ctx, win)
        try:
            trace_extra["activation_select"] = run_select(ctx, win)
        except Exception as e:      # an extra, never the headline
            trace_extra["activation_select"] = {"error": repr(e)}
        try:
            trace_extra["coarse_tracker"] = run_tracker()
        except Exception as e:
            trace_extra["coarse_tracker"] = {"error": repr(e)}
        big_extra = run_config3(args, torch, stream, flush)
        try:
            trace_extra["config5_posegraph"] = run_posegraph()
        except Exception as e:
            trace_extra["config5_posegraph"] = {"error": repr(e)}
        try:
            trace_extra["config4_kitti_loop"] = run_config4(torch)
        except Exception as e:      # an extra, never the headline
            trace_extra["config4_kitti_loop"] = {"error": repr(e)}
    if world > 1 and not use_nccl and ctx.peer_error() != 0:
        raise RuntimeError("peer exchange timed out waiting for a rank")
    strong_extra = None
    if world > 1 and not use_nccl:
        strong_extra = run_config3_sharded(torch, dist, stream, flush, rank, world, local_rank)
    # max over ranks
    if dist is not None:
        tt = torch.tensor([t_ms, t_warm_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_ms, t_warm_ms = float(tt[0]), float(tt[1])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    n_res_rank, n_pts_rank = win.nR, win.nP
    window_its_per_s = args.steps / (t_ms * 1e-3)
    # weak scaling: every rank processes one 8 KF x 2000-point shard per step, so the job processes `world`
    # 2k-point-window iterations per step (units all ranks processed / max-over-ranks time)
    its_per_s = world * window_its_per_s
    hbm_peak, peak_src = peaks()
    b_iter = algorithmic_bytes(n_res_rank, n_pts_rank, NF)   # per GPU (each rank streams its own shard)
    achieved_iter = b_iter / (t_ms * 1e-3 / args.steps) / 1e9
    b_k1 = n_res_rank * (384 + 12 + 12) + n_pts_rank * (80 + 8 + 4)     # SURVEY §8d per-residual / per-point terms
    achieved = b_k1 / (ktimes["k1"] * 1e-6) / 1e9 if ktimes["k1"] > 0 else 0.0
    line = {
        "metric": METRIC, "value": its_per_s, "unit": "GN-iters/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": t_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": common_config(world, full.nP, full.nR),
        "run": {"parallelism": (f"points sharded x{world}, " + ("1 NCCL all-reduce/step" if use_nccl else "1 peer-memory all-reduce kernel/step (NVLink, CUDA IPC), no NCCL in the loop")) if world > 1 else "single GPU",
                "value_unit_note": "value = n_gpus x (GN iterations/s of the sharded window): each rank iterates a 2000-point "
                                   "shard per step; window_iters_per_s is the rate of the whole 2000*n_gpus-point window",
                "l2": "192 MB flush buffer written between timed iterations (inputs 45 MB < 126 MB L2)",
                "timing": "per-iteration CUDA events on the launching stream, summed; max over ranks"},
        "value_l2_warm": world * args.steps / (t_warm_ms * 1e-3),
        "window_iters_per_s": window_its_per_s,
        "wall_ms_per_step_incl_flush": 1e3 * wall / args.steps,
        "roofline": {"bound": "hbm", "kernel": "k1_linearize_accumulate", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                     "frac": achieved / hbm_peak, "traffic": 12254720, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": b_k1, "kernel_us": ktimes,
                     "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of K1, one ncu --set full capture of this workload (profiles/r02z_ncu_full_summary.txt, r02z_gn_ncu_full_raw.csv); bench.py cannot run ncu on itself",
                     "whole_iteration": {"achieved": achieved_iter, "frac": achieved_iter / hbm_peak, "algorithmic_bytes_per_step": b_iter},
                     "note": "2k points: latency-bound, not bandwidth-bound (ideal 0.93 us/iteration); see DESIGN.md §4"},
        "clocks": clocks,
        "gpu_launches": launches,
    }
    if e2e is not None:
        line["e2e"] = e2e
    if trace_extra is not None:
        line["extra_trace_immature"] = trace_extra
    if big_extra is not None:
        line["extra_config3_single_gpu"] = big_extra
    if strong_extra is not None:
        line["extra_config3_sharded"] = strong_extra
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline(win)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(ctx, out_dir):
    """Write what a caller reads back after the last timed Gauss-Newton step (energy, the solved system and update, frame states,
    point depths and steps, residual states and energies) as DIR/<name>.npy in float32 / float64. The window is seeded, so two builds
    run with the same arguments can be compared output for output. With N > 1 ranks this is rank 0's context: energy, lastHS, lastbS,
    lastX and the frame arrays are the whole window's, point_* and residual_* cover rank 0's shard of the points."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"energy": np.array([ctx.energy()[0]])}
    out.update(ctx.last_solution())
    fr = ctx.frames()
    out["frame_state"], out["frame_step"] = fr["state"], fr["step"]
    pts = ctx.points()
    for k in ("idepth", "step", "HdiF", "bdSumF"):
        out["point_" + k] = pts[k]
    res = ctx.residuals(with_J=False)
    for k in ("state_NewState", "state_energy", "state_NewEnergy", "isActive"):
        out["residual_" + k] = res[k]
    for name, a in out.items():
        a = np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float32)
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def run_e2e(ctx, win, args, torch):
    """End to end through the C ABI from HOST buffers (pinned), every step: H2D of the newest keyframe's raw image (+ device
    makeImages), the frame states and the whole window; FullSystem::optimize's prologue + 1 GN iteration; D2H of lastHS / lastbS /
    lastX, energy, point idepth / step / HdiF, residual states + energies. `value` = E2E_CONTEXTS contexts fed round-robin through
    ldso_b200_optimize_from_host_submit / _wait (one window's copies overlap the others' kernels; every step still does all of its copies);
    value_one_context = the same step as ONE blocking call on one context; per_keyframe = one upload + prologue + 6 iterations + one
    read-back per call (what FullSystem::optimize does per keyframe), in GN iterations per second."""
    from ldso_b200 import capi
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
    io = capi.StepIO(ctx, win, pinned_alloc=pin)
    steps = args.steps      # host wall clock over a pipeline: its fill / drain (about one step latency) weighs ~1 / steps in the figure
    for k in range(3):
        io.fused(0, 1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(steps):
        io.fused(0, 1)           # ONE C-ABI call per step: ldso_b200_optimize_from_host
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    # E2E_CONTEXTS contexts fed round-robin from this one host thread: a step's critical path through its stream (uploads -> pyramid ->
    # prologue -> iteration -> read-back, ~270 us) is mostly copy / launch latency, which only other windows in flight can hide
    # (measured, tools/e2e_pipe_prof.py: 1 context 274, 2 contexts 157, 3 contexts 121 us per step; host time of a submit 53 us)
    m = E2E_CONTEXTS
    extra = [capi.Context(win.w, win.h, win.levels, device=torch.cuda.current_device()) for _ in range(m - 1)]
    for c in extra:
        c.load_synth_window(win)
    ios = [io] + [capi.StepIO(c, win, pinned_alloc=pin) for c in extra]
    for k in range(2 * m):
        ios[k % m].fused(0, 1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for k in range(steps):
        if k >= m:
            ios[k % m].wait()            # the step submitted m steps ago on this context: results in the caller's buffers
        ios[k % m].submit(0, 1)
    for k in range(max(steps - m, 0), steps):
        ios[k % m].wait()
    dt_pipe = time.perf_counter() - t0
    # one keyframe's optimize per call: 6 iterations per upload
    for k in range(2):
        io.fused(0, 6)
    t0 = time.perf_counter()
    nkf = 50
    for k in range(nkf):
        io.fused(0, 6)
    dt_kf = time.perf_counter() - t0
    for c in extra:
        c.close()
    return {"value": steps / dt_pipe, "contexts_in_flight": m, "steps": steps, "unit": "GN-iters/s", "h2d_bytes_per_step": int(io.h2d_bytes), "d2h_bytes_per_step": int(io.d2h_bytes),
            "value_one_context": steps / dt,
            "per_keyframe": {"gn_iters_per_s": 6 * nkf / dt_kf, "ms_per_keyframe": 1e3 * dt_kf / nkf, "iterations_per_upload": 6},
            "def": "per step: H2D newest keyframe raw image from pinned memory (+device makeImages), frame states, full window; optimize prologue + "
                   "1 GN iteration; D2H lastHS/lastbS/lastX, energy, point idepth/step/HdiF, residual states+energies; host wall clock. value = "
                   f"{m} contexts fed round-robin from one host thread (ldso_b200_optimize_from_host_submit / _wait: the copies and launches of one window overlap the kernels of the others; every step still does all of its own copies); "
                   "value_one_context = one blocking ldso_b200_optimize_from_host per step; per_keyframe = one upload, prologue + 6 iterations, one read-back"}


def run_config3(args, torch, stream, flush):
    """Not the headline: BASELINE configs[2]'s window (8 KF x 20 000 points, 140 000 residuals) on ONE GPU, to show how the same
    kernels sit against the HBM roofline once the problem is large enough to leave the launch-latency regime."""
    from ldso_b200 import capi, synth
    win = synth.make_window(nF=NF, pts_per_frame=2500, seed=42)
    ctx = capi.Context(win.w, win.h, win.levels, device=torch.cuda.current_device())
    ctx.set_stream(stream.cuda_stream)
    ctx.load_synth_window(win)
    ctx.optimize_begin(want_energy=False)
    for i in range(5):
        ctx.gn_iterations(min(i, 3), 1)
    torch.cuda.synchronize()
    steps = 30
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for k in range(steps):
        flush.fill_(k & 0xff)
        ev[k][0].record(stream); ctx.gn_iterations(3, 1); ev[k][1].record(stream)
    torch.cuda.synchronize()
    t_ms = float(sum(a.elapsed_time(b) for a, b in ev)) / steps
    ctx.kernel_times(True)
    for k in range(20):
        flush.fill_(k & 0xff)
        ctx.gn_iterations(3, 1)
    kt = ctx.kernel_times(False)
    hbm_peak, _ = peaks()
    b_k1 = win.nR * (384 + 12 + 12) + win.nP * (80 + 8 + 4)
    ach = b_k1 / (kt["k1"] * 1e-6) / 1e9 if kt["k1"] > 0 else 0.0
    ctx.close()
    return {"n_points": win.nP, "n_residuals": win.nR, "ms_per_step": t_ms, "gn_iters_per_s": 1e3 / t_ms, "kernel_us": kt,
            "k1_algorithmic_bytes": b_k1, "k1_achieved_GBs": ach, "k1_roofline_frac": ach / hbm_peak}


def _timed_cold_steps(torch, stream, flush, step, steps, dist=None):
    """ms per step of `step()` with the L2 flushed before every step, CUDA events on the launching stream, max over ranks."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    for k in range(steps):
        flush.fill_(k & 0xff)
        ev[k][0].record(stream); step(); ev[k][1].record(stream)
    torch.cuda.synchronize()
    t = float(sum(a.elapsed_time(b) for a, b in ev)) / steps
    if dist is not None:
        tt = torch.tensor([t], device="cuda", dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t = float(tt[0])
    return t


def run_config3_sharded(torch, dist, stream, flush, rank, world, local_rank):
    """BASELINE configs[2]: the FIXED 8 KF x 20 000-point window with its points sharded over the job's GPUs (strong scaling, one
    peer-memory exchange kernel per step), and the same window on rank 0's GPU alone in the same run, so that the line states what
    sharding buys at this point count."""
    from ldso_b200 import capi, synth
    full = synth.make_window(nF=NF, pts_per_frame=2500, seed=42)
    win = synth.shard_window(full, rank, world)
    ctx = capi.Context(win.w, win.h, win.levels, device=local_rank)
    ctx.set_stream(stream.cuda_stream)
    ctx.load_synth_window(win)
    newest = full.nF - 1
    counts = [int(np.sum(synth.shard_window(full, r, world).res_target == newest)) for r in range(world)]
    ctx.set_shard(int(np.sum(counts[:rank])), int(np.sum(counts)))
    handles = [None] * world
    dist.all_gather_object(handles, ctx.peer_export())
    ctx.peer_connect(rank, world, handles)
    dist.barrier()
    ctx.optimize_begin(want_energy=False)
    for i in range(5):
        ctx.gn_iterations(min(i, 3), 1)
    t_sharded = _timed_cold_steps(torch, stream, flush, lambda: ctx.gn_iterations(3, 1), 30, dist)
    err = ctx.peer_error()
    dist.barrier()
    ctx.close()
    t_one = 0.0
    if rank == 0:
        c1 = capi.Context(full.w, full.h, full.levels, device=local_rank)
        c1.set_stream(stream.cuda_stream)
        c1.load_synth_window(full)
        c1.optimize_begin(want_energy=False)
        for i in range(5):
            c1.gn_iterations(min(i, 3), 1)
        t_one = _timed_cold_steps(torch, stream, flush, lambda: c1.gn_iterations(3, 1), 30, None)
        c1.close()
    dist.barrier()
    return {"n_points": int(full.nP), "n_residuals": int(full.nR), "n_gpus": world, "scaling": "strong (fixed window)",
            "ms_per_step_sharded": t_sharded, "gn_iters_per_s_sharded": 1e3 / t_sharded,
            "ms_per_step_one_gpu": t_one, "gn_iters_per_s_one_gpu": (1e3 / t_one) if t_one else None,
            "speedup_vs_one_gpu": (t_one / t_sharded) if t_one else None, "peer_error": int(err),
            "def": "same timing rules as the headline (L2 flushed before every step, CUDA events, max over ranks); one_gpu = the whole window on rank 0's GPU in the same job"}


def run_config4(torch, n_frames=50):
    """BASELINE configs[3]: the tracker + BA LOOP on a synthetic 1232x368 (KITTI-cropped, 5 levels) fly-through, one GPU, through the C
    ABI from host buffers: every frame = raw image H2D + device makeImages + trackNewestCoarse against the newest keyframe; every 5th
    frame = a keyframe: frame states + the whole sliding window (<= 8 KF x 250 points, every point observed in every other keyframe)
    H2D, FullSystem::optimize's prologue + 6 Gauss-Newton iterations + linearizeAll(fix), results D2H, and the tracker's new reference
    (makeCoarseDepthL0 on the device). Host wall clock over the whole loop; the sequence is generated before the clock starts."""
    from ldso_b200 import capi, seq as seqmod
    sq = seqmod.make_sequence(n_frames=n_frames)
    ctx = capi.Context(sq.w, sq.h, sq.levels, device=torch.cuda.current_device())
    pin = [torch.from_numpy(im).pin_memory().numpy() for im in sq.images]
    wins = {k: seqmod.window_arrays(sq, sq.window_kfs(k)) for k in range(0, n_frames, sq.kf_every)}

    def loop():
        ref_k, ref_slot, ref_aff = -1, -1, (0.0, 0.0)
        n_its = n_tracked = n_ok = 0
        t_track = t_ba = t_ba_full = 0.0
        n_full = 0
        errs = []
        aff_est = (0.0, 0.0)
        for k in range(n_frames):
            is_kf = (k % sq.kf_every) == 0
            slot = ((k // sq.kf_every) % 8) if is_kf else 8 + (k & 1)
            ctx.make_images(slot, pin[k])
            if ref_k >= 0:
                t0 = time.perf_counter()
                ctx.tracker_set_frames(ref_aff[0], ref_aff[1], 1.0, slot, 1.0)
                R0, t0v = sq.rel_pose(ref_k, max(k - 1, ref_k))          # zero-velocity model: the previous frame's pose
                ok, R, t, a, b, lr, lf = ctx.tracker_track(R0, t0v, aff_est[0], aff_est[1], sq.levels - 1)
                t_track += time.perf_counter() - t0
                n_tracked += 1; n_ok += int(ok)
                Rg, tg = sq.rel_pose(ref_k, k)
                errs.append(float(np.linalg.norm(t - tg) / max(np.linalg.norm(tg), 1e-9)))
                aff_est = (a, b)
            if is_kf:
                t0 = time.perf_counter()
                kfs = sq.window_kfs(k)
                W = wins[k]
                slots = [((f // sq.kf_every) % 8) for f in kfs]
                ctx.set_frames(W["Rcw"], W["tcw"], W["state_zero"], W["state"], W["ab_exposure"], W["frame_id"], slots, sq.K)
                ctx.set_window(W["pt_host"], W["pt_u"], W["pt_v"], W["pt_idepth"], W["pt_idepth_zero"], W["pt_has_prior"], W["pt_color"],
                               W["pt_weights"], W["res_begin"], W["res_target"])
                if len(kfs) > 1:
                    ctx.optimize_begin(want_energy=False)
                    ctx.gn_iterations(0, 6)
                    n_its += 6
                    ctx.linearize_all(True)                       # FullSystem::optimize ends with linearizeAll(true) (FullSystem.cc:843)
                    res = ctx.residuals_light()
                    pts = ctx.points()
                    newest = len(kfs) - 1
                    m = (W["res_target"] == newest) & (res["state_state"] == capi.RES_IN) & (res["isActive"] == 1)
                    rp = np.repeat(np.arange(len(W["pt_host"])), np.diff(W["res_begin"]))
                    ctx.tracker_make_k(*[float(x) for x in sq.K])
                    ctx.tracker_make_coarse_depth(slot, res["centerProjectedTo"][m], pts["HdiF"][rp[m]])
                else:                                             # the first keyframe: its own points seed the reference (the initializer's job in LDSO)
                    ctx.tracker_make_k(*[float(x) for x in sq.K])
                    ctx.tracker_make_coarse_depth(slot, np.stack([W["pt_u"], W["pt_v"], W["pt_idepth"]], 1), np.full(len(W["pt_u"]), 1e-3, np.float32))
                ref_k, ref_slot = k, slot
                ref_aff = (float(sq.aff[k, 0]), float(sq.aff[k, 1]))
                aff_est = ref_aff
                t_ba += time.perf_counter() - t0
                if len(kfs) == sq.window:
                    t_ba_full += time.perf_counter() - t0; n_full += 1
        return n_its, n_tracked, n_ok, t_track, t_ba, errs, t_ba_full, n_full

    loop()                                   # warm-up pass (allocations, graph capture for every window topology)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n_its, n_tracked, n_ok, t_track, t_ba, errs, t_ba_full, n_full = loop()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    ctx.close()
    n_kf = (n_frames + sq.kf_every - 1) // sq.kf_every
    return {"frames": n_frames, "keyframes": n_kf, "image": f"{sq.w}x{sq.h}, {sq.levels} levels", "frames_per_s": n_frames / dt,
            "gn_iters_per_s_in_loop": n_its / dt, "ms_per_tracked_frame": 1e3 * t_track / max(n_tracked, 1), "ms_per_keyframe_ba": 1e3 * t_ba / n_kf,
            "ms_per_keyframe_ba_full_window": (1e3 * t_ba_full / n_full) if n_full else None,
            "gn_iterations": n_its, "tracked": n_tracked, "tracking_ok": n_ok, "median_translation_err_rel": float(np.median(errs)) if errs else None,
            "def": "host wall clock over 50 frames: per frame raw image H2D + device makeImages + trackNewestCoarse (zero-velocity start) against the newest "
                   "keyframe; every 5th frame a keyframe: frame states + sliding window (<= 8 KF x 250 points) H2D, optimize prologue + 6 GN iterations + "
                   "linearizeAll(fix), point / residual results D2H, makeCoarseDepthL0 on the device; second pass of the same sequence (first pass warms up)"}


def run_posegraph():
    """BASELINE configs[4] (not the headline): Sim(3) pose-graph optimisation, 5000 keyframes / 10 000 loop edges (+ the odometry edges
    to the previous two keyframes), 25 Gauss-Newton rounds as Map.cc:141, through the C ABI from host arrays (uploads and read-back
    inside the timed call). CPU side: the oracle's linearisation of one round (numeric Jacobians, vectorised numpy, one core); its
    sparse direct solve of this graph does not finish within minutes (the random loop edges fill the factor in), so only that part is
    timed and said so."""
    from ldso_b200 import capi
    from oracle import posegraph as pg
    g = pg.make_graph(5000, 10000, seed=0)
    ctx = capi.Context(64, 64, 1)
    ctx.posegraph_optimize(g["q"], g["t"], g["ei"], g["ej"], g["mq"], g["mt"], g["info"], g["fixed"], iterations=2)      # warm-up
    t0 = time.perf_counter()
    q, t, chi, ncg = ctx.posegraph_optimize(g["q"], g["t"], g["ei"], g["ej"], g["mq"], g["mt"], g["info"], g["fixed"], iterations=25, pcg_tol=1e-10)
    dt = time.perf_counter() - t0
    ctx.close()
    t0 = time.perf_counter()
    pg.linearize(g["q"], g["t"], g["ei"], g["ej"], g["mq"], g["mt"], g["info"])
    dto = time.perf_counter() - t0
    return {"keyframes": 5000, "edges": int(len(g["ei"])), "gn_rounds": 25, "seconds": dt, "ms_per_round": 1e3 * dt / 25, "cg_iterations_total": int(ncg),
            "chi2_first": float(chi[0]), "chi2_last": float(chi[-1]), "max_translation_err_vs_truth": float(np.abs(t - g["gt"]).max()),
            "cpu_oracle_linearize_ms_per_round_1core": 1e3 * dto,
            "def": "ldso_b200_posegraph_optimize: warp-per-edge numeric-Jacobian linearisation + block-Jacobi PCG (relative residual 1e-10) + oplus, 25 rounds, host arrays in/out; "
                   "cpu figure = the oracle's linearisation alone (its sparse direct solve of this graph does not finish within 10 minutes)"}


def _trace_inputs(win):
    from ldso_b200 import synth
    case = synth.make_trace_case(win, 250, seed=5, hosts=range(win.nF - 2))          # 1500 candidates, what LDSO keeps per frame
    return case


def run_trace(ctx, win):
    """SURVEY 8f rank 2 (not the headline metric): one FullSystem::traceNewCoarse pass = ImmaturePoint::traceOn of 1500 candidates on
    the newest keyframe, through the C ABI from host arrays (uploads, kernel, read-back inside the timed region)."""
    case = _trace_inputs(win)
    init = {k: [] for k in ("color", "weights", "gradH", "energyTH")}
    for h in range(win.nF - 2):
        m = case.host == h
        r = ctx.immature_init(h, case.u[m], case.v[m])
        for k in init:
            init[k].append(r[k])
    init = {k: np.concatenate(v) for k, v in init.items()}
    n = case.n
    new = win.nF - 1

    def fresh():
        return dict(u=case.u, v=case.v, host=case.host, **init, idepth_min=np.zeros(n, np.float32), idepth_max=np.full(n, np.nan, np.float32),
                    quality=np.full(n, 10000.0, np.float32), status=np.full(n, 5, np.int32), uv=np.zeros((n, 2), np.float32),
                    interval=np.zeros(n, np.float32))
    for _ in range(3):
        ctx.trace_immature(new, fresh(), case.KRKi[new], case.Kt[new], case.aff[new])
    reps = 20
    states = [fresh() for _ in range(reps)]
    t0 = time.perf_counter()
    for p in states:
        ctx.trace_immature(new, p, case.KRKi[new], case.Kt[new], case.aff[new])
    dt = (time.perf_counter() - t0) / reps
    return {"candidates": n, "ms_per_pass": 1e3 * dt, "candidates_per_s": n / dt, "good": int((states[-1]["status"] == 0).sum()),
            "def": "ImmaturePoint::traceOn of 1500 fresh candidates (unbounded idepth interval: full epipolar search) on one frame, host arrays in/out"}


def run_tracker():
    """SURVEY 8 rows b1-b4 (not the headline metric): one CoarseTracker::trackNewestCoarse (coarse-to-fine LM over all pyramid levels,
    calcRes + calcGSSSE per evaluation) of a 640x480 frame against a reference keyframe, through the C ABI, images resident; the oracle
    port on one host core beside it (the reference's tracker is single-threaded)."""
    from tests import oracle_py
    from ldso_b200 import capi, synth
    pair = synth.make_track_pair()
    ot = oracle_py.OracleTracker(pair, fast=True)
    ctx = capi.Context(pair.w, pair.h, pair.levels)
    ctx.upload_frame(0, pair.ref_pyr)
    ctx.upload_frame(1, pair.new_pyr)
    ctx.tracker_make_k(*[float(x) for x in pair.K])
    for l in range(pair.levels):
        ctx.tracker_set_ref_level(l, *ot.pc(l))
    ctx.tracker_set_frames(pair.ref_aff[0], pair.ref_aff[1], 1.0, 1, 1.0)
    I, z = np.eye(3), np.zeros(3)
    for _ in range(3):
        r = ctx.tracker_track(I, z, 0.0, 0.0, pair.levels - 1)
    reps = 20
    t0 = time.perf_counter()
    for _ in range(reps):
        r = ctx.tracker_track(I, z, 0.0, 0.0, pair.levels - 1)
    dt = (time.perf_counter() - t0) / reps
    t0 = time.perf_counter()
    ro = ot.track(I, z, 0.0, 0.0, pair.levels - 1)
    dto = time.perf_counter() - t0
    # FullSystem::trackNewCoarse's hypothesis loop as one launch: identity + the 26 small rotations (rotDelta = 0.02, FullSystem.cc:300-330)
    rd = 0.02
    hyp = [np.zeros(3)] + [np.array(v, float) * rd for v in ((1, 0, 0), (0, 1, 0), (0, 0, 1), (-1, 0, 0), (0, -1, 0), (0, 0, -1), (1, 1, 0), (0, 1, 1), (1, 0, 1),
                                                                  (-1, 1, 0), (0, -1, 1), (-1, 0, 1), (1, -1, 0), (0, 1, -1), (1, 0, -1), (-1, -1, 0), (0, -1, -1), (-1, 0, -1),
                                                                  (-1, -1, -1), (-1, -1, 1), (-1, 1, -1), (-1, 1, 1), (1, -1, -1), (1, -1, 1), (1, 1, -1), (1, 1, 1))]
    Rs = np.stack([synth.so3_exp(h) for h in hyp]); ts = np.zeros((len(hyp), 3)); af = np.zeros((len(hyp), 2), np.float32)
    for _ in range(3):
        bres = ctx.tracker_track_batch(Rs, ts, af, pair.levels - 1)
    t0 = time.perf_counter()
    for _ in range(reps):
        bres = ctx.tracker_track_batch(Rs, ts, af, pair.levels - 1)
    dtb = (time.perf_counter() - t0) / reps
    # one calcRes + calcGSSSE evaluation at level 0 against the HBM roofline (SURVEY 8d: pc_n (16 + 48) + 624 bytes)
    n0 = len(ot.pc(0)[0])
    for _ in range(5):
        ctx.tracker_eval(0, pair.R_true, pair.t_true, 0.0, 0.0, 20.0)
    t0 = time.perf_counter()
    for _ in range(100):
        ctx.tracker_eval(0, pair.R_true, pair.t_true, 0.0, 0.0, 20.0)
    dte = (time.perf_counter() - t0) / 100
    hbm_peak, _ = peaks()
    eval_bytes = n0 * 64 + 624
    ctx.close()
    ref_ms = None
    try:                                   # the reference's own CoarseTracker.cc (oracle/_ref/libref_ba.so), when it is there
        if oracle_py.ref_lib() is not None:
            ref_ms = 1e3 * oracle_py.RefTracker(pair).track(I, z, 0.0, 0.0, pair.levels - 1, reps=10)[5]
    except Exception:
        ref_ms = None
    return {"ms_per_track": 1e3 * dt, "tracks_per_s": 1.0 / dt,
            "batch": {"hypotheses": len(hyp), "ms_per_batch": 1e3 * dtb, "ms_per_hypothesis": 1e3 * dtb / len(hyp), "ok": int(bres["ok"].sum()),
                      "def": "ldso_b200_tracker_track_batch: FullSystem::trackNewCoarse's 27 starting poses (identity + 26 rotations of 0.02 rad) in one launch, one CTA each, host arrays in/out"},
            "roofline": {"bound": "hbm", "kernel": "k_trk_eval (calcRes + calcGSSSE, level 0)", "algorithmic_bytes_per_launch": eval_bytes, "pc_n": n0,
                         "us_per_call_through_c_abi": 1e6 * dte, "achieved": eval_bytes / dte / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": eval_bytes / dte / 1e9 / hbm_peak,
                         "note": "one evaluation moves ~0.6 MB: launch + synchronise + 624-byte read-back dominate; the call is latency-bound by construction"}, "reference_ms_per_track_1core": ref_ms, "cpu_port_ms_per_track_1core": 1e3 * dto,
            "calcRes_evaluations": int(ro[-1]),
            "converged": bool(r[0]), "same_outcome_as_cpu_port": bool(r[0] == ro[0]),
            "translation_err_rel": float(np.linalg.norm(r[2] - pair.t_true) / max(np.linalg.norm(pair.t_true), 1e-12)),
            "def": "trackNewestCoarse from the identity on synth.make_track_pair() (640x480, all levels), pose in / pose out through the C ABI"}


def run_select(ctx, win):
    """SURVEY 8f rank 2, last piece: FullSystem::activatePointsMT's selection (CoarseDistanceMap + the order-dependent greedy pass) for
    the traced candidates of the bench window, through the C ABI from host arrays; the oracle port's time beside it."""
    from tests import oracle_py
    from ldso_b200 import capi
    ctx = capi.Context(win.w, win.h, win.levels)       # a fresh context: the bench context's window has been optimised, the oracle's has not
    ctx.load_synth_window(win)
    case = _trace_inputs(win)
    tr = oracle_py.OracleTrace(win, case)
    tr.trace_on(win.nF - 2); tr.trace_on(win.nF - 1)
    newest = win.nF - 1
    m = case.host != newest
    n = int(m.sum())
    quality = np.where(np.isfinite(tr.quality[m]), tr.quality[m], 0).astype(np.float32)
    a = (case.u[m], case.v[m], case.host[m], tr.idepth_min[m], tr.idepth_max[m], tr.status[m], tr.interval[m], quality, np.ones(n, np.float32))
    for _ in range(3):
        act = ctx.select_activation(newest, 2.0, *a)
    reps = 20
    t0 = time.perf_counter()
    for _ in range(reps):
        act = ctx.select_activation(newest, 2.0, *a)
    dt = (time.perf_counter() - t0) / reps
    o = oracle_py.OracleBA(win, threads_mode=1, fast=True)      # -O3 -march=native: the timing build (its FMA contraction may move a projection across a pixel boundary)
    t0 = time.perf_counter()
    o.select_activation(newest, 2.0, *a)
    dto = time.perf_counter() - t0
    ao, _ = oracle_py.OracleBA(win, threads_mode=1).select_activation(newest, 2.0, *a)      # the bit-reproducible build: the checker
    ctx.close()
    return {"candidates": n, "window_points": int(win.nP), "ms_per_call": 1e3 * dt, "cpu_port_ms_per_call_1core": 1e3 * dto, "selected": int((act == 1).sum()),
            "identical_to_cpu_port": bool(np.array_equal(act, ao)),
            "def": "distance map of the window's points at level 1 + greedy accept/keep/delete pass, currentMinActDist = 2, host arrays in/out"}


def cpu_baseline(win):
    from tests import oracle_py
    o = oracle_py.OracleBA(win, threads_mode=6, fast=True)
    o.optimize_begin()
    for i in range(3):
        o.gn_iteration(i)
    sec = o.time_gn(40, 3)
    case = _trace_inputs(win)
    tr = oracle_py.OracleTrace(win, case)
    t0 = time.perf_counter()
    tr.trace_on(win.nF - 1)
    trace_ms = 1e3 * (time.perf_counter() - t0)
    sec_ref = _ref_arm_seconds_per_iter(40, 6)
    if sec_ref:
        return {"trace_immature_ms_per_pass_1core": trace_ms,
                "value": 1.0 / sec_ref, "unit": "GN-iters/s", "cores": 6, "kind": "reference", "port_value": 1.0 / sec,
                "sample": f"40 full GN iterations of the same 8 KF x 2000 point window by the reference's own back-end translation units "
                          f"(oracle/_ref/libref_ba.so: compiled -O3 -march=native against stand-in Eigen headers, FullSystem's driver loop "
                          f"restated), 6 worker threads = reference NUM_THREADS, host has {os.cpu_count()} cores; port_value = median of 40 by "
                          f"the oracle port"}
    return {"trace_immature_ms_per_pass_1core": trace_ms,
            "value": 1.0 / sec, "unit": "GN-iters/s", "cores": 6, "kind": "port",
            "sample": f"median of 40 full GN iterations of the same 8 KF x 2000 point window; oracle port "
                      f"(g++ -O3 -march=native), 6 worker threads = reference NUM_THREADS, host has {os.cpu_count()} cores"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl"], help="N>1: device-side peer-memory exchange (default) or NCCL all-reduce")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
