#!/usr/bin/env python
"""bench.py -- replans/sec of FUEL's per-replan hot path on B200 (BASELINE.json metric).

One step = one replan = {ESDF update over the whole map} + {frontier sweep + clustering +
PCA split over the same box} + {B trajectories x K cost/gradient evaluations, mask
NORMAL_PHASE|MINTIME} on BASELINE config 2 (office.pcd 200x120x40 @0.1 m, B = 1024,
20 control points).  N GPUs = N independent planners (one process per GPU, no data-path
collective; scaling = weak), value = replans of all ranks / max-over-ranks device time.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--evals 64] [--batch 1024] [--no-esdf512] [--dump-outputs DIR]

--impl reference times the CPU restatement of the reference (oracle/, all host threads)
on the same workload; the unmodified reference cannot be built here (ROS1/Eigen3/PCL/NLopt
absent, see DESIGN.md).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "replans_per_sec"
UNIT = "replans/s"


def profile_traffic(key):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture) of the
    named kernel/stage, read from the committed summary profiles/traffic.json (written by tools/ncu_traffic.py from
    the .ncu-rep); None if that stage has no capture."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        v = d.get(key)
        return float(v["bytes"]) if v else None
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.dev = dev
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for k, nm in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_workload(batch, seed_offset=0, workload="office"):
    from fuel_b200 import workloads as W
    g, inflate = W.office3_map() if workload == "office3" else W.office_map()
    tri = W.office_known(g, inflate)
    tr = W.make_trajectories(g, inflate, B=batch, n_pts=20, seed=20260922 + seed_offset)
    return g, inflate, tri, tr


# --------------------------------------------------------------------------------------------
# reference arm: the oracle (CPU restatement of the reference) on all host threads
# --------------------------------------------------------------------------------------------
def cpu_replan_setup(batch):
    import oracle
    g, inflate, tri, tr = build_workload(batch)
    og = oracle.make_grid(g.n, g.res, g.origin, g.box_min, g.box_max)
    B = batch
    tcs = oracle.traj_consts(B)
    for b in range(B):
        oracle.fill_traj_const(tcs[b], tr["pt_dist"][b], tr["dt"][b], tr["start"][b], tr["end_pos"][b][None, :])
    from fuel_b200 import workloads as W
    x = W.pack_x(tr["ctrl"], tr["dt"])
    return dict(oracle=oracle, g=g, og=og, inflate=inflate, tri=tri, tcs=tcs, x=x, B=B)


def cpu_replan(S, evals, threads, bspline_only=False):
    """One replan on the CPU (oracle port).  Returns per-stage seconds.  ESDF lines and trajectories go over
    `threads` OpenMP threads; the frontier BFS is single-threaded as in the reference."""
    oracle = S["oracle"]
    g = S["g"]
    t0 = time.perf_counter()
    if not bspline_only or "dist" not in S:
        S["dist"] = oracle.update_esdf3d(S["og"], S["inflate"], S["tri"], [0, 0, 0], np.array(g.n) - 1, True, False,
                                         threads=threads)
    dist = S["dist"]
    t1 = time.perf_counter()
    ncl = 0
    if not bspline_only:
        flag = np.zeros(g.n, dtype=np.int8)
        ncl = len(oracle.frontier_search(S["og"], S["tri"], flag, g.origin, g.map_max, oracle.frontier_params()))
    t2 = time.perf_counter()
    mask = oracle.NORMAL_PHASE | oracle.MINTIME
    x = S["x"]
    xb, fb, ne = oracle.optimize_batch(S["og"], dist, oracle.opt_params(), S["tcs"], 20, mask, x, max_eval=evals,
                                       xtol_rel=0.0, threads=threads)
    t3 = time.perf_counter()
    return dict(esdf=t1 - t0, frontier=t2 - t1, bspline=t3 - t2, total=t3 - t0, n_clusters=ncl,
                evals_min=int(ne.min()), evals_mean=float(ne.mean()))


# the reference's own code (oracle/_ref/libfuel_ref.so: its sdf_map.cpp, frontier_finder.cpp, bspline_optimizer.cpp
# compiled unmodified in the build container; prebuilt here) -- used for the CPU numbers whenever it is present
REF_OPT = dict(ld_smooth=20.0, ld_dist=10.0, ld_feasi=2.0, ld_start=100.0, ld_end=0.5, ld_guide=1.5, ld_waypt=0.3,
               ld_view=0.0, ld_time=1.0, dist0=0.7, max_vel=2.0, max_acc=2.0, dlmin=0.0, wnl=0.0, max_iteration_num1=2,
               max_iteration_num2=2000, max_iteration_num3=200, max_iteration_num4=200, max_iteration_time1=0.0001,
               max_iteration_time2=0.005, max_iteration_time3=0.003, max_iteration_time4=0.003, algorithm1=15,
               algorithm2=11, bspline_degree=3)  # exploration_manager/launch/algorithm.xml:170-192


class _Quiet:
    """The reference prints to std::cout from its hot path; keep bench.py's stdout to the one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        self._null = os.open(os.devnull, os.O_WRONLY)
        os.dup2(self._null, 1)

    def __exit__(self, *a):
        os.dup2(self._saved, 1)
        os.close(self._null)
        os.close(self._saved)


def ref_available():
    import oracle
    oracle.build()
    return oracle.ref_raycast() is not None


def ref_replan_setup(batch, evals):
    """The same workload on the reference's own classes (the office map is centred, as SDFMap::initMap requires)."""
    import oracle
    g, inflate, tri, tr = build_workload(batch)
    size = np.array(g.n) * g.res
    assert np.allclose(np.asarray(g.origin)[:2], -size[:2] / 2)
    params = dict(resolution=g.res, map_size_x=size[0], map_size_y=size[1], map_size_z=size[2], ground_height=g.origin[2],
                  obstacles_inflation=0.199, local_bound_inflate=0.5, local_map_margin=50, default_dist=0.0, optimistic=1,
                  signed_dist=0, p_hit=0.65, p_miss=0.35, p_min=0.12, p_max=0.90, p_occ=0.80, max_ray_length=4.5,
                  virtual_ceil_height=-10.0)
    for ax, lo, hi in zip("xyz", g.box_min, g.box_max):
        params["box_min_" + ax], params["box_max_" + ax] = float(lo), float(hi)
    with _Quiet():
        ref = oracle.RefSDFMap(**params)
    assert ref.n == tuple(g.n)
    lg = lambda p: float(np.log(p / (1 - p)))  # noqa: E731
    ref.inflate[:] = inflate.reshape(-1)
    ref.occupancy[:] = np.where(tri == 0, lg(0.12) - 0.01, np.where(tri == 2, lg(0.90), lg(0.12))).reshape(-1)
    ref.set_modes(1, 0)
    ref.set_local_bound((0, 0, 0), np.array(g.n) - 1)
    with _Quiet():
        ff = oracle.RefFrontierFinder(ref, dict(top_angle=0.56125, left_angle=0.69222, right_angle=0.68901, max_dist=4.5,
                                                vis_dist=1.0),
                                      cluster_min=100, cluster_size_xy=2.0, cluster_size_z=10.0, min_candidate_dist=0.75,
                                      min_candidate_clearance=0.21, candidate_dphi=15 * 3.1415926 / 180.0, candidate_rmax=2.5,
                                      candidate_rmin=1.5, candidate_rnum=3, down_sample=3, min_visib_num=15,
                                      min_view_finish_fraction=0.2)
    from fuel_b200 import workloads as W
    x = W.pack_x(tr["ctrl"], tr["dt"])
    rng = np.random.default_rng(5)
    # the K-1 further points at which the objective is evaluated: small steps around the start, like a line search
    probes = x[:, None, :] + rng.normal(size=(batch, evals - 1, x.shape[1])) * 0.03
    probes[:, :, -1] = np.abs(probes[:, :, -1]) + 1e-3
    return dict(oracle=oracle, g=g, ref=ref, ff=ff, tr=tr, probes=np.ascontiguousarray(probes), B=batch)


def ref_replan(S, evals, threads, bspline_only=False):
    """One replan on the reference's own code: updateESDF3d, searchFrontiers (both single-threaded as written),
    K combineCost calls per trajectory over `threads` threads (one BsplineOptimizer each)."""
    oracle, g, ref, ff, tr = S["oracle"], S["g"], S["ref"], S["ff"], S["tr"]
    with _Quiet():
        t0 = time.perf_counter()
        if not bspline_only or not S.get("esdf_done"):
            ref.update_esdf3d()
            S["esdf_done"] = True
        t1 = time.perf_counter()
        if not bspline_only:
            ff.flags[:] = 0
            ref.R.ref_map_set_updated_box(ref.h, oracle._p(np.asarray(g.origin, dtype=np.float64)),
                                          oracle._p(np.asarray(g.map_max, dtype=np.float64)))
            ref.R.ref_ff_search(ff.h)
        t2 = time.perf_counter()
        mask = oracle.NORMAL_PHASE | oracle.MINTIME
        oracle.ref_combine_cost_batch(ref, REF_OPT, tr["ctrl"], tr["dt"], mask, tr["start"], tr["end_pos"],
                                      S["probes"][:, :evals - 1], threads=threads)
        t3 = time.perf_counter()
        ncl = ref.R.ref_ff_count(ff.h, 0)
    return dict(esdf=t1 - t0, frontier=t2 - t1, bspline=t3 - t2, total=t3 - t0, n_clusters=ncl,
                evals_min=evals, evals_mean=float(evals))


def physical_cores():
    """Physical cores this process may run on (SMT siblings counted once)."""
    try:
        allowed = os.sched_getaffinity(0)
    except AttributeError:
        allowed = set(range(os.cpu_count() or 1))
    seen = set()
    for c in allowed:
        try:
            sib = open("/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list" % c).read().strip()
        except OSError:
            sib = str(c)
        seen.add(sib)
    return max(1, len(seen))


def calibrate_threads(fn, S, evals, ncores):
    """Thread count of the trajectory batch: the candidate with the best MEDIAN of 3 timings of the B-spline stage
    alone (ESDF/frontier are single-threaded in the reference and must not vote), never above the physical cores."""
    cands = sorted({c for c in (ncores, ncores // 2, ncores // 4, 64, 32, 16, 8, 4, 2, 1) if 1 <= c <= ncores},
                   reverse=True)
    table = {}
    for c in cands:
        fn(S, min(evals, 8), c, bspline_only=True)
        table[c] = float(np.median([fn(S, evals, c, bspline_only=True)["bspline"] for _ in range(3)]))
    best = min(table, key=lambda c: table[c])
    return best, {str(c): round(1e3 * v, 3) for c, v in table.items()}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")  # idle OpenMP workers must not spin beside the 1-thread BFS
    ncpu = os.cpu_count() or 1
    use_ref = ref_available()
    if use_ref:
        S = ref_replan_setup(args.batch, args.evals)
        cpu_replan = ref_replan  # noqa: F811  (the port below is the fallback when oracle/_ref was not built)
    else:
        S = cpu_replan_setup(args.batch)
        cpu_replan = globals()["cpu_replan"]
    # "all the host threads it can use": the trajectory batch goes over OpenMP threads; on a many-core host the
    # small batch stops scaling long before all cores are busy, so the count is calibrated (median of 3 runs of
    # the B-spline stage per candidate, capped at the physical cores) and reported as `cores`.
    threads, calib = calibrate_threads(cpu_replan, S, args.evals, physical_cores())
    for _ in range(args.warmup):
        cpu_replan(S, args.evals, threads)
    t0 = time.perf_counter()
    stages = []
    for _ in range(args.steps):
        stages.append(cpu_replan(S, args.evals, threads))
    dt = time.perf_counter() - t0
    val = args.steps / dt
    line = {
        "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "impl": "reference",
        "config": workload_config(args),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "reference" if use_ref else "port",
                         "sample": ("%d full replans on the reference's own code (oracle/_ref: sdf_map.cpp, frontier_finder.cpp, "
                                    "bspline_optimizer.cpp compiled unmodified): updateESDF3d and searchFrontiers single-threaded "
                                    "as written, B=%d trajectories x K=%d combineCost evaluations over %d threads with one "
                                    "BsplineOptimizer each (NLopt itself absent: the objective is evaluated at K points)"
                                    % (args.steps, args.batch, args.evals, threads)) if use_ref else
                                   ("%d full replans (B=%d x K=%d evals each), OpenMP over ESDF lines and "
                                    "trajectories, frontier BFS single-threaded as in the reference"
                                    % (args.steps, args.batch, args.evals))},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "stage_ms": {k: 1e3 * float(np.mean([s[k] for s in stages])) for k in ("esdf", "frontier", "bspline")},
        "cores": threads, "cores_physical": physical_cores(), "cores_logical": ncpu,
        "thread_calibration_bspline_ms": calib,
        "evals_done_min": min(s["evals_min"] for s in stages),
        "n_planners": 1,
        "note": "ONE CPU planner on rank 0 regardless of --gpus (the reference is one process); at N > 1 the driver's "
                "ratio therefore compares N GPU planners with one CPU planner",
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(args):
    return {"workload": "office.pcd 200x120x40 @0.1m (BASELINE config 2): full-box optimistic ESDF update + "
                        "frontier sweep/cluster/split + %d-trajectory x 20 ctrl-pt B-spline batch, %d "
                        "cost/gradient evaluations per trajectory" % (args.batch, args.evals),
            "batch": args.batch, "ctrl_pts": 20, "evals_per_replan": args.evals,
            "cost_mask": "SMOOTHNESS|DISTANCE|FEASIBILITY|START|END|MINTIME",
            "parallelism": "replica x%d (independent planners, no collective)" % args.gpus,
            "l2": "256 MB L2 flush between timed steps (flush time excluded: each step has its own event pair)",
            "overlap": "frontier search (own stream, begin/end) runs beside ESDF update + solver"
                       if not getattr(args, "no_overlap", False) else "stages run back to back"}


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
class GpuPlanner:
    def __init__(self, dev, batch, evals, seed_offset=0, overlap=True, workload="office"):
        import ctypes as C

        import torch

        import fuel_b200
        from fuel_b200 import workloads as W
        from fuel_b200._lib import FuelTrajConst
        self.C, self.torch, self.fuel = C, torch, fuel_b200
        self.dev = dev
        self.evals = evals
        g, inflate, tri, tr = build_workload(batch, seed_offset, workload)
        self.g = g
        self.B = batch
        m = fuel_b200.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max, optimistic=True, device=dev)
        m.occupancy_buffer_inflate_[...] = inflate
        m.setOccupancyBuffer(tristate=tri)
        self.m = m
        env = fuel_b200.EDTEnvironment()
        env.setMap(m)
        self.ff = fuel_b200.FrontierFinder(env)
        self.opt = fuel_b200.BsplineOptimizer()
        self.opt.setEnvironment(env)
        self.mask = self.opt.NORMAL_PHASE | self.opt.MINTIME
        self.x_host = W.pack_x(tr["ctrl"], tr["dt"])
        self.tcs = self.opt.traj_consts_from_arrays(tr["pt_dist"], tr["dt"], tr["start"], tr["end_pos"])
        self.nvar = self.x_host.shape[1]
        # resident copies for the HBM-resident timing
        # a dedicated (non-default) stream: the library runs on it and the events are recorded on it
        self.stream = torch.cuda.Stream(device=dev)
        torch.cuda.set_stream(self.stream)
        m.set_stream(self.stream.cuda_stream)
        tcb = np.frombuffer(self.tcs, dtype=np.uint8)
        self.d_tc = torch.from_numpy(tcb.copy()).to("cuda:%d" % dev)
        self.d_x = torch.from_numpy(self.x_host).to("cuda:%d" % dev)
        self.d_xw = torch.empty_like(self.d_x)
        self.d_n = torch.empty(batch, dtype=torch.int32, device="cuda:%d" % dev)
        from fuel_b200._lib import FuelSolveParams
        self.sp = FuelSolveParams()
        # the metric's unit of work is B x K combineCost evaluations (the CPU arms do exactly K): xtol off and the
        # solver restarts instead of stopping when a line search fails or the gradient vanishes
        self.sp.max_eval, self.sp.lbfgs_m, self.sp.xtol_rel, self.sp.flags = evals, 6, 0.0, 1
        self.d_f = torch.empty(batch, dtype=torch.float64, device="cuda:%d" % dev)
        self.d_g = torch.empty((batch, self.nvar), dtype=torch.float64, device="cuda:%d" % dev)
        self.pin_x = torch.from_numpy(self.x_host).pin_memory()
        self.pin_f = torch.empty(batch, dtype=torch.float64).pin_memory()
        self.pin_g = torch.empty((batch, self.nvar), dtype=torch.float64).pin_memory()
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda:%d" % dev)
        m.upload()
        m.pin(self.x_host)
        self._tcs_view = np.frombuffer(self.tcs, dtype=np.uint8)
        m.pin(self._tcs_view)
        self.clusters, self.n_clusters = [], 0
        # result buffers of the optimiser, reused every replan (the reference keeps best_variable_ as a member)
        self.opt_out = (np.empty_like(self.x_host), np.empty(batch, dtype=np.float64), np.empty(batch, dtype=np.int32))
        # the frontier subsystem has its own stream in the library: the search is enqueued first
        # (fuelgpu_frontier_search_begin), the ESDF update and the solver run beside it on the main
        # stream, and the result is collected last (fuelgpu_frontier_search_end)
        self.overlap = overlap
        # issue order inside an overlapped replan: the frontier search goes first -- its 8-CTA cluster kernel needs whole
        # SMs and does not get them once the solver's 256 CTAs are resident (measured: it then runs AFTER the solver,
        # 0.72 ms per replan instead of 0.40).  FUELGPU_BENCH_ORDER=solver_first shows it.
        self.solver_first = os.environ.get("FUELGPU_BENCH_ORDER", "frontier_first") == "solver_first"

    def _frontier_begin(self):
        self.ff.reset_flags()
        self.ff.search_box_begin(self.g.origin, self.g.map_max)

    def _frontier_end(self):
        self.clusters = self.ff.search_box_end()
        self.n_clusters = len(self.clusters)

    def l2_flush(self):
        self.flush.zero_()

    def replan_resident(self):
        """Inputs already in HBM: occupancy byte, x, trajectory constants."""
        L, C = self.fuel.lib(), self.C
        if not (self.overlap and self.solver_first):
            self._frontier_begin()
        if not self.overlap:
            self._frontier_end()
        self.m.updateESDF3d()
        h = self.m.handle
        # the solver loop of BsplineOptimizer::optimize() on the device: K = max_eval cost/gradient
        # evaluations per trajectory inside one persistent kernel
        self.d_xw.copy_(self.d_x, non_blocking=True)
        rc = L.fuelgpu_bspline_optimize_batch_dev(h, self.B, 20, self.mask, C.byref(self.opt.params_),
                                                  C.c_void_p(self.d_tc.data_ptr()), C.byref(self.sp),
                                                  C.c_void_p(self.d_xw.data_ptr()), C.c_void_p(self.d_f.data_ptr()),
                                                  C.c_void_p(self.d_n.data_ptr()))
        if rc:
            raise RuntimeError(L.fuelgpu_last_error(h))
        if self.overlap:
            if self.solver_first:
                self._frontier_begin()
            self._frontier_end()

    def replan_e2e(self):
        """Through the reference-facing host API with HOST buffers: occupancy H2D, ESDF update,
        ESDF D2H (the host mirror SDFMap::getDistance readers need), frontier search + fetch,
        and BsplineOptimizer::optimize()'s solver loop on the device (x and the trajectory constants
        H2D once, best x / cost / eval count D2H once)."""
        m = self.m
        m.upload(wait=not self.overlap)  # overlap: the mirrors are not touched before the final synchronize()
        if not (self.overlap and self.solver_first):
            self._frontier_begin()
        if not self.overlap:
            out = self.ff.search_box_end()
        m.updateESDF3d()
        if self.overlap:
            # solver enqueued (its inputs go H2D beside the ESDF kernels), then the D2H mirror copy, which runs beside
            # the solver; the frontier result is marshalled on the host meanwhile
            self.opt.optimizeBatchBegin(self.x_host, self.tcs, 20, self.mask, self.evals, xtol_rel=0.0, exact_evals=True)
            if self.solver_first:
                self._frontier_begin()
            m.download(wait=False)
            out = self.ff.search_box_end()
            x, f, ne = self.opt.optimizeBatchEnd(out=self.opt_out)
            m.synchronize()  # ESDF host mirror complete
        else:
            m.download(wait=True)
            x, f, ne = self.opt.optimizeBatch(self.x_host, self.tcs, 20, self.mask, self.evals, xtol_rel=0.0,
                                              out=self.opt_out, exact_evals=True)
        self.last_neval = ne
        return out, f

    def dump_outputs(self, out_dir, max_traj=32768):
        """What the last resident replan handed back -- the ESDF, the frontier clusters, and the solver's best
        variables, costs and evaluation counts -- as out_dir/<name>.npy in float32 / float64 (integers are exact in
        float64), about 4.5 MB at the default batch.  Above max_traj trajectories the solver's outputs are a fixed
        seeded sample of them (traj_index), which keeps the whole dump under 64 MB."""
        os.makedirs(out_dir, exist_ok=True)
        self.torch.cuda.synchronize(self.dev)
        cl = self.clusters
        rows = np.arange(self.B)
        if self.B > max_traj:
            rows = np.sort(np.random.default_rng(0).choice(self.B, max_traj, replace=False))

        def cat(arrays, empty_shape):
            return np.concatenate(arrays).astype(np.float64) if arrays else np.zeros(empty_shape)

        out = {
            "esdf": self.m.download(dtype=np.float32),                                     # [nx, ny, nz] metres
            "traj_index": rows.astype(np.float64),
            "x_best": self.d_xw.cpu().numpy()[rows],                                       # [B, 3 * 20 + 1]
            "f_best": self.d_f.cpu().numpy()[rows],                                        # [B]
            "n_eval": self.d_n.cpu().numpy()[rows].astype(np.float64),                     # [B]
            "frontier_cell_offsets": np.cumsum([0] + [c.cells_addr_.size for c in cl]).astype(np.float64),
            "frontier_cells": cat([c.cells_addr_ for c in cl], (0,)),                       # voxel addresses, BFS order
            "frontier_filtered_offsets": np.cumsum([0] + [len(c.filtered_cells_) for c in cl]).astype(np.float64),
            "frontier_filtered": cat([np.reshape(c.filtered_cells_, (-1, 3)) for c in cl], (0, 3)),
            "frontier_average": cat([np.reshape(c.average_, (1, 3)) for c in cl], (0, 3)),
            "frontier_box_min": cat([np.reshape(c.box_min_, (1, 3)) for c in cl], (0, 3)),
            "frontier_box_max": cat([np.reshape(c.box_max_, (1, 3)) for c in cl], (0, 3)),
        }
        for k, v in out.items():
            np.save(os.path.join(out_dir, k + ".npy"), v)

    def e2e_bytes(self):
        nv = self.g.nvox
        from fuel_b200._lib import FuelTrajConst
        h2d = 2 * nv + self.x_host.nbytes + self.B * (FuelTrajConst.guide.offset + 4)
        d2h = 4 * nv + self.B * 12 + self.x_host.nbytes
        return h2d, d2h


def esdf512_roofline(dev, peak, peak_src, variant="V1", reps=5):
    """The north-star roofline kernel: full ESDF rebuild of pillar.pcd (V1, tiled) on 512^3.
    Algorithmic bytes = 5 B/voxel (1 B occupancy in + 4 B fp32 distance out, SURVEY 8d)."""
    import torch

    import fuel_b200
    from fuel_b200 import workloads as W
    g, inflate = W.pillar_map(variant)
    m = fuel_b200.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max, optimistic=True, device=dev)
    m.occupancy_buffer_inflate_[...] = inflate
    m.occupancy_tri_[...] = np.where(inflate == 1, 2, 1).astype(np.uint8)
    m.upload()
    st = torch.cuda.current_stream(dev)
    assert st.cuda_stream != 0, "events must be recorded on the stream the kernels run on"
    m.set_stream(st.cuda_stream)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda:%d" % dev)
    ms = []
    for i in range(reps + 2):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        m.updateESDF3d()
        e1.record(st)
        torch.cuda.synchronize(dev)
        if i >= 2:
            ms.append(e0.elapsed_time(e1))
    m.close()
    t = float(np.mean(ms)) * 1e-3
    alg = 5.0 * g.nvox
    ach = alg / t / 1e9
    return {"kernel": "esdf_update 512^3 (zpack_kernel + per z chunk: envelope_tile_kernel zy, envelope_tile_kernel x)",
            "bound": "hbm",
            "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
            # DRAM read+write of all kernels of one update, ncu --set full (profiles/traffic.json)
            "traffic": profile_traffic("esdf512_" + variant.lower()),
            "algorithmic_bytes": alg, "ms": 1e3 * t, "peak_source": peak_src,
            "workload": "pillar.pcd %s on 512^3 @0.1m, optimistic, full rebuild (box = whole map); "
                        "L2 flushed before every timed update" % ("V1 (tiled to fill the cube)" if variant == "V1"
                                                                  else "V0 (file as is, mostly empty cube)")}


def frontier512_roofline(dev, peak, peak_src, reps=4):
    """BASELINE config 3, second half: the frontier sweep + clustering + split over the 512^3 pillar map (V1, seeded
    known region).  Algorithmic bytes = 2 B/voxel (tri-state read + frontier_flag_ read-modify-write, SURVEY 8d)."""
    import torch

    import fuel_b200
    from fuel_b200 import workloads as W
    g, inflate = W.pillar_map("V1")
    tri = W.known_region(g, inflate, seed=7, n_poses=64, radius=4.5)
    m = fuel_b200.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max, device=dev)
    m.occupancy_buffer_inflate_[...] = inflate
    m.setOccupancyBuffer(tristate=tri)
    m.upload()
    env = fuel_b200.EDTEnvironment()
    env.setMap(m)
    ff = fuel_b200.FrontierFinder(env)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda:%d" % dev)
    ms, wall = [], []
    ncl = ncell = 0
    for i in range(reps + 1):
        ff.reset_flags()
        flush.zero_()
        m.synchronize()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        out = ff.search_box(g.origin, g.map_max)
        t1 = time.perf_counter()
        if i >= 1:
            ms.append(m.last_timing()["frontier"])
            wall.append(1e3 * (t1 - t0))
        ncl, ncell = len(out), int(sum(c.cells_addr_.size for c in out))
    # the voxel sweep alone (the HBM-bound part: occupancy byte + frontier_flag_ byte per voxel): classification,
    # scan of the per-CTA counts and ordered compaction, as fuelgpu_frontier_candidates runs them
    sweep_ms, ncand = [], 0
    for i in range(reps + 1):
        ff.reset_flags()
        flush.zero_()
        m.synchronize()
        torch.cuda.synchronize(dev)
        addr, _ = ff.candidates(g.origin, g.map_max, 0, g.n[2] - 1)
        ncand = int(addr.size)
        if i >= 1:
            sweep_ms.append(m.last_timing()["frontier"])
    m.close()
    t = float(np.mean(ms)) * 1e-3
    ts = float(np.mean(sweep_ms)) * 1e-3
    alg = 2.0 * g.nvox
    ach = alg / t / 1e9
    return {"kernel": "frontier_search 512^3 (classify sweep + union-find + claims + level-synchronous PCA split)",
            "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
            "traffic": profile_traffic("frontier512"), "algorithmic_bytes": alg, "ms": 1e3 * t,
            "sweep": {"kernel": "classify_words_kernel + scan + compact_words_kernel (fuelgpu_frontier_candidates, whole z "
                                "range; includes the host read of the candidate count between scan and compaction)",
                      "ms": 1e3 * ts, "achieved": alg / ts / 1e9, "frac": alg / ts / 1e9 / peak, "unit": "GB/s",
                      "algorithmic_bytes": alg, "n_candidates": ncand},
            "wall_ms_incl_fetch": float(np.mean(wall)), "n_clusters": ncl, "n_cells": ncell, "peak_source": peak_src,
            "workload": "pillar.pcd V1 on 512^3 @0.1m, known region = 64 seeded 4.5 m balls, frontier_flag_ reset, search "
                        "box = whole map; device time of the frontier stream (events), L2 flushed before every search"}


def sharded_esdf_arm(local, rank, world, reps=5):
    """BASELINE config 4: synthetic 1024x1024x256 map, z-sharded ESDF over all ranks (fuelgpu_sharded_esdf_*,
    NCCL called inside the library).  Collective: every rank calls it.  Device time = max over ranks.  Also runs
    the parity check of the sharded path against the single-GPU kernel on a smaller map (the driver's pytest box
    has one GPU), and times the same update on ONE rank (a 1-rank communicator on rank 0) for reference."""
    import torch
    import torch.distributed as dist

    import fuel_b200
    from fuel_b200 import workloads as W
    from fuel_b200.dist import ShardedESDF
    dev = "cuda:%d" % local
    out = {}
    # ---- parity: sharded == single GPU, voxel for voxel (finite values to 1e-6 relative, same +inf set) ----
    # (x lines of 1024 samples: the x tiles are the 2-CTA cluster form reading their rows as `world` pieces)
    npar = (1024, 96, 32 * world)
    g, inflate = W.random_boxes_map(n=npar, seed=11, n_boxes=48, ground_idx=3)
    sh = ShardedESDF(npar, g.res, optimistic=True, device=local)
    z0, z1 = sh.z_range()
    occ = torch.from_numpy(((inflate[:, :, z0:z1] << 2) | 1).astype(np.uint8)).contiguous().to(dev)
    slab = sh.update(occ)
    full = sh.gather_full(slab).cpu().numpy()
    m = fuel_b200.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max, optimistic=True, device=local)
    m.occupancy_buffer_inflate_[...] = inflate
    m.occupancy_tri_[...] = 1
    m.upload()
    m.updateESDF3d()
    ref = m.download().copy()
    fin = np.isfinite(ref)
    ok = bool(np.array_equal(np.isinf(full), ~fin) and np.allclose(full[fin], ref[fin], rtol=1e-6, atol=0))
    # one planner, G GPUs (SURVEY 8e row 3): the gathered field installed in a second map, the trajectory batch split
    # over the ranks, results gathered -- must equal the whole batch solved on this rank's own ESDF, bit for bit
    from fuel_b200.dist import optimize_batch_split
    m2 = fuel_b200.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max, optimistic=True, device=local)
    sh.gather_into_map(slab, m2)
    tr = W.make_trajectories(g, inflate, B=96, n_pts=20, seed=31)
    x0 = W.pack_x(tr["ctrl"], tr["dt"])
    ok_split = True
    res = []
    for mm in (m, m2):
        env = fuel_b200.EDTEnvironment()
        env.setMap(mm)
        opt = fuel_b200.BsplineOptimizer()
        opt.setEnvironment(env)
        tcs = opt.traj_consts_from_arrays(tr["pt_dist"], tr["dt"], tr["start"], tr["end_pos"])
        mask = opt.NORMAL_PHASE | opt.MINTIME
        if mm is m:
            res.append(tuple(a.copy() for a in opt.optimizeBatch(x0, tcs, 20, mask, 32)))
        else:
            res.append(optimize_batch_split(opt, x0, tcs, 20, mask, 32))
    ok_split = all(np.array_equal(a, b) for a, b in zip(res[0], res[1]))
    m.close()
    m2.close()
    sh.close()
    flag = torch.tensor([1 if ok else 0, 1 if ok_split else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out["parity_vs_single_gpu"] = {"map": list(npar), "ok_all_ranks": bool(int(flag[0].item()) == 1),
                                   "split_batch_equals_whole_batch": bool(int(flag[1].item()) == 1)}
    # ---- timing on the config-4 map ----
    n = (1024, 1024, 256)
    g, inflate = W.random_boxes_map(n=n, seed=11, n_boxes=4096)
    sh = ShardedESDF(n, g.res, optimistic=True, device=local)
    z0, z1 = sh.z_range()
    occ = torch.from_numpy(((inflate[:, :, z0:z1] << 2) | 1).astype(np.uint8)).contiguous().to(dev)
    st = torch.cuda.current_stream(local)
    buf = torch.empty((n[0], n[1], sh.nzl), dtype=torch.float32, device=dev)
    for _ in range(3):
        sh.update(occ, out=buf)
    torch.cuda.synchronize(local)
    ms, stages = [], []
    for _ in range(reps):
        dist.barrier()
        torch.cuda.synchronize(local)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        sh.update(occ, out=buf)
        e1.record(st)
        torch.cuda.synchronize(local)
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms.append(float(t.item()))
        stages.append(sh.last_timing())
    sent = sh.bytes_exchanged()
    p2p = sh.uses_peer_memory()
    sh.close()
    out.update({"map": list(n), "n_gpus": world,
                "exchange": ("peer memory: the zy tile kernels store the int32 partial straight into the destination rank's "
                             "buffer over NVLink (CUDA IPC), one 4 B/rank all-gather as the barrier") if p2p else
                            "ncclSend/ncclRecv rounds on a second stream", "ms": float(np.median(ms)), "ms_all": [round(v, 3) for v in ms],
                "stage_ms_rank0": {k: round(float(np.median([s_[k] for s_ in stages])), 3) for k in stages[0]},
                "bytes_sent_per_rank": sent, "voxels": int(np.prod(n)),
                "note": "device time of one whole-map update, max over ranks; stages: occupancy all-to-all (1 B/voxel), "
                        "z records + zy tiles with the int32 partial's exchange rounds running beside them, wait for the "
                        "last rounds, x tiles"})
    # ---- the same update on ONE GPU (rank 0, 1-rank communicator) ----
    solo = dist.new_group([0]) if world > 1 else None  # collective over the default group
    if rank == 0:
        sh1 = ShardedESDF(n, g.res, optimistic=True, device=local, group=solo)
        occ1 = torch.from_numpy(((inflate << 2) | 1).astype(np.uint8)).contiguous().to(dev)
        buf1 = torch.empty(n, dtype=torch.float32, device=dev)
        for _ in range(2):
            sh1.update(occ1, out=buf1)
        torch.cuda.synchronize(local)
        m1 = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            sh1.update(occ1, out=buf1)
            e1.record(st)
            torch.cuda.synchronize(local)
            m1.append(e0.elapsed_time(e1))
        sh1.close()
        out["ms_1gpu"] = float(np.median(m1))
        del occ1, buf1
    if world > 1:
        dist.barrier()
    return out


def config5_arm(local, rank, world, args, steps=10):
    """BASELINE config 5: office3.pcd 200x300x40, one independent planner per GPU, 4096-trajectory batch each -- the same
    resident replan (ESDF update + frontier search + K evaluations per trajectory in the device solver) as the metric,
    on the bigger map and batch.  Collective-safe: every rank reaches the all_reduce whatever happened before it."""
    import torch
    import torch.distributed as dist
    ms, info = float("nan"), {}
    try:
        P5 = GpuPlanner(local, 4096, args.evals, seed_offset=100 * rank, overlap=not args.no_overlap, workload="office3")
        for _ in range(3):
            P5.l2_flush()
            P5.replan_resident()
        torch.cuda.synchronize(local)
        evs, stage = [], {"esdf": [], "frontier": [], "bspline": []}
        for _ in range(steps):
            P5.l2_flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(P5.stream)
            P5.replan_resident()
            e1.record(P5.stream)
            evs.append((e0, e1))
            t = P5.m.last_timing()
            for k in stage:
                stage[k].append(t[k])
        torch.cuda.synchronize(local)
        ms = sum(a.elapsed_time(b) for a, b in evs)
        nev = P5.d_n.cpu().numpy()
        info = {"stage_ms": {k: float(np.median(v)) for k, v in stage.items()}, "evals_done_min": int(nev.min()),
                "n_frontier_clusters": P5.n_clusters, "voxels": int(P5.g.nvox)}
        P5.m.close()
    except Exception as e:  # noqa: BLE001
        info = {"error": repr(e)}
    t = torch.tensor([ms if ms == ms else 1e30], dtype=torch.float64, device="cuda:%d" % local)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    mx = float(t.item())
    out = {"workload": "office3.pcd 200x300x40 @0.1m, %d independent planner(s), 4096-trajectory x 20 ctrl-pt batch each, "
                       "%d evaluations per trajectory, inputs resident" % (world, args.evals),
           "steps": steps}
    out.update(info)
    if mx < 1e29:
        out.update({"value": world * steps / (mx * 1e-3), "unit": UNIT, "ms_per_step": mx / steps})
    return out


def next_rows_timing(dev):
    """SURVEY 8f rows built on top of the hot path, timed beside it (not part of the metric): one fused depth
    frame (proessDepthImage + inputPointCloud), clearAndInflateLocalMap, and sampleViewpoints for the clusters of
    the office replan -- wall time per call through the host API, and the oracle's single-thread time."""
    import fuel_b200
    import oracle
    from fuel_b200 import workloads as W
    g, inflate = W.office_map()
    tri = W.office_known(g, inflate)
    og = oracle.make_grid(g.n, g.res, g.origin, g.box_min, g.box_max)
    out = {}
    m = fuel_b200.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max, device=dev)
    m.setFusionParams()
    frames = []
    for i in range(4):
        cam = np.array([0.25 * i, 0.1 * i, 1.0])
        img, R = W.depth_image(g, inflate, cam, 0.8 * i)
        m.pin(img)
        frames.append((img, R, cam))
    for img, R, cam in frames:
        m.inputDepthImage(img, R, cam)
    m.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        for img, R, cam in frames:
            m.inputDepthImage(img, R, cam)
    m.synchronize()
    out["fusion_depth_frame_ms"] = 1e3 * (time.perf_counter() - t0) / 20
    for _ in range(3):  # warm-up: the first call pays lazy allocations and page-locking of the mirror
        m.clearAndInflateLocalMap()
    m.synchronize()
    t0 = time.perf_counter()
    for _ in range(10):
        m.clearAndInflateLocalMap()
    m.synchronize()
    out["inflate_local_map_ms"] = 1e3 * (time.perf_counter() - t0) / 10
    fus = oracle.Fusion(og, oracle.fusion_params())
    cp = oracle.camera_params()
    t0 = time.perf_counter()
    for img, R, cam in frames:
        fus.input_point_cloud(oracle.process_depth_image(cp, img, R, cam), cam)
    out["cpu_fusion_depth_frame_ms"] = 1e3 * (time.perf_counter() - t0) / len(frames)
    m.close()
    m = fuel_b200.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max, optimistic=True, device=dev)
    m.occupancy_buffer_inflate_[...] = inflate
    m.setOccupancyBuffer(tristate=tri)
    m.upload()
    env = fuel_b200.EDTEnvironment()
    env.setMap(m)
    ff = fuel_b200.FrontierFinder(env)
    ftrs = ff.search_box(g.origin, g.map_max)
    ff.sampleViewpointsRaw(ftrs)
    t0 = time.perf_counter()
    for _ in range(10):
        ff.sampleViewpointsRaw(ftrs)
    out["sample_viewpoints_ms"] = 1e3 * (time.perf_counter() - t0) / 10
    vp = oracle.view_params()
    t0 = time.perf_counter()
    for f in ftrs:
        oracle.sample_viewpoints(og, tri, inflate, vp, f.average_, f.filtered_cells_)
    out["cpu_sample_viewpoints_ms"] = 1e3 * (time.perf_counter() - t0)
    out["n_clusters"] = len(ftrs)
    m.close()
    return out


def bind_near_gpu(local):
    """Pin this process to the CPUs NVML lists as local to its GPU (same NUMA node / PCIe root): with one process per
    GPU the host side of a replan (launches, pinned-buffer copies, result marshalling) otherwise runs wherever the
    launcher left it.  FUELGPU_BENCH_BIND=0 disables it.  Returns the number of CPUs in the new set, or None."""
    if os.environ.get("FUELGPU_BENCH_BIND", "1") == "0":
        return None
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        uuid = "GPU-" + str(torch.cuda.get_device_properties(local).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return None


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libfuelgpu has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    cpus_bound = bind_near_gpu(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    P = GpuPlanner(local, args.batch, args.evals, seed_offset=100 * rank, overlap=not args.no_overlap)
    st = P.stream

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(local)

    for _ in range(max(args.warmup, 3)):
        P.l2_flush()
        P.replan_resident()
    torch.cuda.synchronize(local)

    # ---- resident timing: K steps, each with its own event pair; L2 flushed in between ----
    sampler = ClockSampler(local)
    stage = {"esdf": [], "frontier": [], "bspline": []}
    launches0 = P.m.launch_count()
    barrier()
    sampler.start()
    wall0 = time.perf_counter()
    evs = []
    for _ in range(args.steps):
        P.l2_flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        P.replan_resident()
        e1.record(st)
        evs.append((e0, e1))
        t = P.m.last_timing()
        for k in stage:
            stage[k].append(t[k])
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    launches = P.m.launch_count() - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    nev = P.d_n.cpu().numpy()  # evaluations the solver actually performed in the last timed replan
    evals_min, evals_mean = int(nev.min()), float(nev.mean())
    if evals_min != args.evals:
        raise SystemExit("bench.py: the solver stopped after %d < %d evaluations on some trajectory -- the unit of work "
                         "of the metric (B x K combineCost) was not performed" % (evals_min, args.evals))
    if args.dump_outputs and rank == 0:
        P.dump_outputs(args.dump_outputs)
    tt = torch.tensor([dev_ms], dtype=torch.float64, device="cuda:%d" % local)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    max_ms = float(tt.item())
    value = world * args.steps / (max_ms * 1e-3)

    # ---- end-to-end timing through the host API (host buffers, copies inside) ----
    for _ in range(2):
        P.replan_e2e()
    barrier()
    e2e0 = time.perf_counter()
    ee = []
    for _ in range(args.steps):
        P.l2_flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        P.replan_e2e()
        e1.record(st)
        ee.append((e0, e1))
    barrier()
    e2e_wall = time.perf_counter() - e2e0
    e2e_ms = sum(a.elapsed_time(b) for a, b in ee)
    t2 = torch.tensor([e2e_ms], dtype=torch.float64, device="cuda:%d" % local)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_val = world * args.steps / (float(t2.item()) * 1e-3)
    h2d, d2h = P.e2e_bytes()

    # ---- BASELINE config 4 (z-sharded ESDF over all ranks) beside the replica metric, N > 1 only ----
    sharded = None
    if world > 1 and not args.no_sharded:
        try:
            sharded = sharded_esdf_arm(local, rank, world)
        except Exception as e:  # noqa: BLE001
            sharded = {"error": repr(e)}

    config5 = None if args.no_config5 else config5_arm(local, rank, world, args, steps=args.steps)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = load_peaks()
    st_ms = {k: float(np.mean(v)) for k, v in stage.items()}
    # dominant stage of the replan and its roofline.  The B-spline batch is latency / L2-gather
    # bound (SURVEY 8d): its HBM fraction is reported for completeness, from the algorithmic
    # 1624 B per trajectory-evaluation; the ESDF rows use 5 B/voxel; frontier 2 B/voxel.
    alg = {"esdf": 5.0 * P.g.nvox, "frontier": 2.0 * P.g.nvox, "bspline": 1624.0 * args.batch}
    alg["bspline"] *= evals_mean  # one launch = K evaluations of the batch (K checked against the solver's own count)
    per_launch_ms = dict(st_ms)
    dom = max(("esdf", "frontier", "bspline"), key=lambda k: st_ms[k])
    ach = alg[dom] / (per_launch_ms[dom] * 1e-3) / 1e9
    notes = {
        "bspline": "dominant stage of the office replan: the solver is dependent-latency-bound (1 warp per trajectory), "
                   "the 3.8 MB ESDF is L2-resident, so the HBM fraction is reported for completeness only",
        "frontier": "dominant stage of the office replan: the frontier search of a 0.96 M-voxel map is launch/barrier-"
                    "latency-bound (2 B/voxel = 1.9 MB, L2-resident), so the HBM fraction is reported for completeness "
                    "only; the HBM-bound frontier case is roofline_frontier512",
        "esdf": "dominant stage of the office replan: a 0.96 M-voxel map is L2-resident and launch-latency-bound; the "
                "HBM-bound ESDF case is roofline_esdf512"}
    roofline = {"kernel": {"esdf": "esdf_update (zpack + envelope tiles)", "frontier": "frontier_search (sweep + clustering)",
                           "bspline": "optimize_gram_kernel<6> (persistent L-BFGS solver: K evaluations of the batch in one launch)"}[dom],
                "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": profile_traffic("office_" + dom), "algorithmic_bytes": alg[dom],
                "peak_source": peak_src, "note": notes[dom]}
    extra = {}
    if not args.no_esdf512 and world == 1:
        try:
            extra["roofline_esdf512"] = esdf512_roofline(local, peak, peak_src, "V1")
            extra["roofline_esdf512_v0"] = esdf512_roofline(local, peak, peak_src, "V0")
        except Exception as e:  # noqa: BLE001
            extra["roofline_esdf512"] = {"error": repr(e)}
        try:
            extra["roofline_frontier512"] = frontier512_roofline(local, peak, peak_src)
        except Exception as e:  # noqa: BLE001
            extra["roofline_frontier512"] = {"error": repr(e)}

        try:
            extra["next_rows"] = next_rows_timing(local)
        except Exception as e:  # noqa: BLE001
            extra["next_rows"] = {"error": repr(e)}

    # ---- CPU baseline, 1 thread (the reference is single-threaded): its own code when oracle/_ref is present ----
    use_ref = ref_available()
    if use_ref:
        S = ref_replan_setup(args.batch, args.evals)
        cpu_fn = ref_replan
    else:
        S = cpu_replan_setup(args.batch)
        cpu_fn = cpu_replan
    cpu_fn(S, 2, 1)
    t0 = time.perf_counter()
    nrep = 0
    cst = []
    while nrep < 3 or (time.perf_counter() - t0 < 12 and nrep < 50):
        cst.append(cpu_fn(S, args.evals, 1))
        nrep += 1
    cpu_dt = time.perf_counter() - t0
    cpu_val = nrep / cpu_dt

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": max_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64 (cost/gradient), i32+f32 (ESDF), u8 (frontier)",
        "data": "synthetic (voxelised office.pcd fixture, seeded known region and trajectories)",
        "config": workload_config(args),
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "wall_ms_per_step": 1e3 * e2e_wall / args.steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": {"value": cpu_val, "unit": UNIT, "cores": 1, "kind": "reference" if use_ref else "port",
                         "sample": ("%d full replans of the same workload on 1 host thread through the reference's own code "
                                    "(oracle/_ref: its sdf_map.cpp / frontier_finder.cpp / bspline_optimizer.cpp compiled "
                                    "unmodified; K combineCost evaluations per trajectory)" % nrep) if use_ref else
                                   ("%d full replans of the same workload on 1 host thread (the reference is "
                                    "single-threaded; its two ros::Time::now() calls per combineCost omitted)" % nrep),
                         "stage_ms": {k: 1e3 * float(np.mean([s[k] for s in cst])) for k in
                                      ("esdf", "frontier", "bspline")}},
        "stage_ms": {"esdf": st_ms["esdf"], "frontier": st_ms["frontier"], "bspline": st_ms["bspline"]},
        "wall_ms_per_step": 1e3 * wall / args.steps,
        "n_frontier_clusters": P.n_clusters,
        "evals_done_min": evals_min, "evals_done_mean": evals_mean,
    }
    if cpus_bound is not None:
        line["host_cpus_bound_near_gpu"] = cpus_bound
    line.update(extra)
    if sharded is not None:
        line["sharded_esdf"] = sharded
    if config5 is not None:
        line["config5_office3_b4096"] = config5
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--evals", type=int, default=64)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--no-esdf512", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="skip the config-4 z-sharded ESDF arm at N > 1")
    ap.add_argument("--no-config5", action="store_true", help="skip the office3 / 4096-trajectory replan (BASELINE config 5)")
    ap.add_argument("--no-overlap", action="store_true", help="run the frontier search after the ESDF update instead of beside it")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last resident replan "
                    "computed (ESDF, frontier clusters, solver results) to DIR/<name>.npy; rank 0 only")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
