#!/usr/bin/env python3
"""bench.py -- headline benchmark of the ICP hot path (BASELINE.json config 2).

Workload (SURVEY.md 8d, config 2): point-to-plane ICP, 1M -> 1M synthetic points + analytic
normals (surface z = 0.1 sin 4pi x cos 4pi y), max_correspondence_distance 0.02,
ICPConvergenceCriteria(0, 0, 30): exactly 30 updates / 31 searches per registration.

  step            = one RegistrationICP call (index build + source ordering + 31 fused launches)
  value           = ICP iterations / s, clouds resident in HBM when the timed region starts
  e2e.value       = the same through the public API with HOST (pinned) buffers: H2D of both clouds
                    and D2H of the result inside the timed region
  roofline        = algorithmic bytes of the fused iteration kernel (36 B / source point,
                    SURVEY.md 8d) / mean device time of one fused iteration = CUDA events around
                    the launch loop / number of iterations (so the idle instance, the fixed-order
                    sum and the solve are charged to the kernel: a conservative figure)
  cpu_baseline    = the CPU oracle port (kd-tree + OpenMP, all host cores) on the same workload
  --impl reference= that CPU implementation timed as its own arm

N > 1 (torchrun): the source is split into contiguous blocks of its Hilbert order, one per rank, the
target and its index are replicated, and the 32 partial sums are exchanged once per iteration (peer-
memory mailboxes over NVLink fused into the launch's tail; --comm nccl for ncclAllReduce): strong
scaling of the same 1M -> 1M problem.  Sub-records: certificates_off and config3 (N = 1), config4
(Generalized ICP 5M -> 5M, the configuration BASELINE names for 8 GPUs) at every N, config5
(Colored-ICP pyramid on a 20M-point pair) at N = 1.
"""
import argparse
import ctypes as C
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

ALG_BYTES_PER_POINT = 36  # src xyz 12 + matched target xyz 12 + matched normal 12 (SURVEY.md 8d)
MAX_DIST = 0.02
ITERS = 30
WORKLOAD = "config2: point-to-plane ICP 1M->1M + normals, 30 iters, r=0.02 (SURVEY.md 8d)"
DUMP_BYTES = 64 << 20  # --dump-outputs: at most this much in all


def result_arrays(T, fitness, inlier_rmse, correspondence_set):
    """what a caller of registration_icp receives (RegistrationResult), as float64 arrays for --dump-outputs"""
    return {"transformation": np.asarray(T, np.float64).reshape(4, 4), "fitness": np.float64(fitness),
            "inlier_rmse": np.float64(inlier_rmse), "correspondence_set": np.asarray(correspondence_set, np.float64)}


def dump_outputs(path, arrays):
    """Writes each array as path/<name>.npy.  Should the arrays exceed DUMP_BYTES, every array with more rows than
    its share keeps a fixed, seeded sample of its rows (ascending), and <name>_rows.npy holds their indices."""
    os.makedirs(path, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in list(arrays.items()):
        if total > DUMP_BYTES and a.ndim > 0 and a.nbytes > DUMP_BYTES // (2 * len(arrays)):
            keep = max(1, DUMP_BYTES // (2 * len(arrays)) // (a.nbytes // len(a)))
            rows = np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))
            arrays[name], arrays[name + "_rows"] = a[rows], rows.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region.  NVML (pynvml) when importable -- a sample costs
    microseconds, so even a 100 ms timed region gets tens of samples -- else nvidia-smi."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.maxclk = None
        self.recording = False          # samples are kept only while the timed region runs
        self.ready = threading.Event()  # NVML initialised (nvmlInit takes a driver lock for tens of ms:
                                        # it must not happen inside the timed region)

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        self.maxclk = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        self.ready.set()
        while not self.stop_flag:
            if self.recording:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for name, bit in self.REASONS.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
            time.sleep(0.005)

    def _run_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        self.ready.set()
        while not self.stop_flag:
            if not self.recording:
                time.sleep(0.005)
                continue
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.maxclk = float(f[1])
                for nme, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(nme)
            except Exception:
                pass
            time.sleep(0.2)

    def run(self):
        try:
            self._run_nvml()
        except Exception:
            self._run_smi()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.maxclk, "reasons": sorted(self.reasons),
                "samples": len(s)}


def measured_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the fused kernel, from the committed ncu
    capture of this workload (profiles/roofline_traffic.json); None if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


def make_workload(n):
    from cupoch_b200.testing import datagen
    tgt, tn = datagen.surface(n, 11)
    src = datagen.make_source(tgt, datagen.gt_transform(), 13, 14, 5e-4)
    return src, tgt, tn


def cpu_threads():
    """threads for the CPU arm: every core this process may run on.  Set explicitly -- torchrun exports
    OMP_NUM_THREADS=1, which would silently turn the 'all host cores' baseline into a single-thread one."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except Exception:
        n = max(1, os.cpu_count() or 1)
    # a container may see every core of the host but be limited by a cgroup CPU quota: more threads than the quota
    # only adds contention (the round-1 CPU arm varied 8x between two "128-core" boxes)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()[:2]
        if q != "max":
            n = max(1, min(n, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def cpu_arm(src, tgt, tn, runs=3, budget_s=30.0, warm=0):
    """The oracle port of cupoch's RegistrationICP (kd-tree + OpenMP) on the host cores: `runs` full registrations
    (kd-tree build included), median time; stops early once budget_s is spent.  Returns (median seconds, all
    seconds, last result, info)."""
    from oracle import oracle_py as orc
    L = orc.lib()
    n_thr = cpu_threads()
    L.orc_set_num_threads(n_thr)

    def step():
        return orc.registration_icp(orc.P2PLANE, src, tgt, MAX_DIST, tgt_nrm=tn, relative_fitness=0, relative_rmse=0,
                                    max_iteration=ITERS)
    for _ in range(warm):
        step()
    times, r, t_all = [], None, time.perf_counter()
    for _ in range(max(1, runs)):
        t0 = time.perf_counter()
        r = step()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_all > budget_s:
            break
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = None
    info = {"threads": orc.num_threads(), "nproc": os.cpu_count(), "affinity": aff,
            "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS"), "runs_s": [round(t, 3) for t in times]}
    return float(np.median(times)), times, r, info


def run_reference(args, rank):
    """CPU arm: the oracle port of cupoch's RegistrationICP (kd-tree + OpenMP) on ALL host cores (rank 0 only)."""
    if rank != 0:
        return
    src, tgt, tn = make_workload(args.points)
    med, times, r, info = cpu_arm(src, tgt, tn, runs=args.steps, budget_s=float("inf"), warm=min(args.warmup, 1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, result_arrays(r["transformation"], r["fitness"], r["inlier_rmse"], r["correspondence_set"]))
    v = ITERS / med
    print(json.dumps({
        "impl": "reference", "metric": "icp_iterations_per_sec", "value": v, "unit": "iter/s", "n_gpus": args.gpus,
        "steps": len(times), "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * med, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "points": args.points, "iterations": ITERS,
                   "step": "one RegistrationICP call incl. index (kd-tree) build; median of the timed steps"},
        "cpu_baseline": {"value": v, "unit": "iter/s", "cores": info["threads"], "kind": "port",
                         "sample": "full workload: %d registrations x %d iterations, kd-tree build included, median" % (len(times), ITERS),
                         **info},
        "e2e": {"value": v, "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "final_fitness": r["fitness"], "final_rmse": r["inlier_rmse"],
    }))


def pinned_array(L, shape):
    nbytes = int(np.prod(shape)) * 4
    p = L.cphb_malloc_host(nbytes)
    buf = (C.c_float * (nbytes // 4)).from_address(p)
    return np.frombuffer(buf, dtype=np.float32).reshape(shape), p


def run_native(args, rank, world):
    import cupoch_b200 as cph
    from cupoch_b200 import _lib
    from cupoch_b200.utility import DeviceArray, as_f16
    L = _lib.lib()
    _lib.require_gpu()
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    _lib.check(L.cphb_set_device(local_rank))
    comm = None
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        from cupoch_b200.distributed import make_comm
        comm_kind = args.comm
        try:
            comm = make_comm(dist, rank, world, device="cuda", kind=comm_kind)
        except Exception as e:  # make_comm fails on every rank together (e.g. CUDA IPC not permitted)
            if comm_kind != "p2p":
                raise
            sys.stderr.write("rank %d: peer-memory exchange unavailable (%s); using NCCL\n" % (rank, e))
            comm_kind = "nccl"
            comm = make_comm(dist, rank, world, device="cuda", kind="nccl")
        args.comm = comm_kind

    n = args.points
    # like the reference's initialize_allocator(PoolAllocation, initial_pool_size): reserve the pool once
    cph.initialize_allocator(initial_pool_size=max(1 << 30, 600 * n))
    src, tgt, tn = make_workload(n)
    from cupoch_b200.distributed import shard_range
    lo, hi = shard_range(n, rank, world)
    # every rank holds the full source; the library keeps this rank's Hilbert-contiguous block of it
    src_local = src
    shard = (rank, world) if world > 1 else None
    R = cph.registration
    est, crit = R.TransformationEstimationPointToPlane(), R.ICPConvergenceCriteria(0, 0, ITERS)
    init = np.eye(4, dtype=np.float32)

    # resident clouds
    s_pc = cph.geometry.PointCloud(src_local)
    t_pc = cph.geometry.PointCloud(tgt)
    t_pc.normals = tn
    flush = DeviceArray((256 << 20,), np.uint8)  # > 126 MB L2

    def barrier():
        _lib.check(L.cphb_stream_synchronize(None))
        if dist is not None:
            dist.barrier()
            import torch
            torch.cuda.synchronize()

    def step_resident():
        return R.registration_icp(s_pc, t_pc, MAX_DIST, init, est, crit, comm=comm, shard=shard)

    ev = [L.cphb_event_create() for _ in range(2)]

    step_log = []

    def timed(fn, steps):
        """sum of per-step device times (CUDA events), L2 flushed between steps outside the timed region"""
        total_ms, last = 0.0, None
        for _ in range(steps):
            _lib.check(L.cphb_memset(flush.ptr, 0, flush.nbytes, None))
            barrier()
            _lib.check(L.cphb_event_record(ev[0], None))
            last = fn()
            _lib.check(L.cphb_event_record(ev[1], None))
            ms = C.c_float(0)
            _lib.check(L.cphb_event_elapsed_ms(ev[0], ev[1], C.byref(ms)))
            total_ms += ms.value
            step_log.append(round(ms.value, 3))
        return total_ms, last

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.ready.wait(timeout=20)
    barrier()   # (ranks finish their set-up at different times; the first exchange of a registration waits for every peer)
    for _ in range(args.warmup):
        step_resident()
    barrier()
    sampler.recording = True
    launches0 = L.cphb_launch_count()
    total_ms, res = timed(step_resident, args.steps)
    resident_steps_ms = list(step_log)
    launches = L.cphb_launch_count() - launches0
    loop_ms, loop_launches = res.loop_ms, res.loop_launches
    if args.dump_outputs:
        corr = res.correspondence_set
        if dist is not None:    # each rank holds the pairs of its block: the caller of N ranks receives all of them
            from cupoch_b200.distributed import gather_correspondences
            corr = gather_correspondences(dist, corr, 0, world)
        outputs = result_arrays(res.transformation, res.fitness, res.inlier_rmse, corr)

    # ---- end-to-end through the public API with host (pinned) buffers ---------------------------
    h_src, p1 = pinned_array(L, src_local.shape)
    h_tgt, p2 = pinned_array(L, tgt.shape)
    h_tn, p3 = pinned_array(L, tn.shape)
    h_src[:], h_tgt[:], h_tn[:] = src_local, tgt, tn
    d2h = [0]

    dbg = os.environ.get("BENCH_DEBUG")

    def step_e2e():
        t0 = time.perf_counter()
        s2 = cph.geometry.PointCloud(h_src)         # H2D (pinned)
        t2 = cph.geometry.PointCloud(h_tgt)
        t2.normals = h_tn
        if dbg:
            L.cphb_stream_synchronize(None)
            sys.stderr.write("e2e upload %.3f ms\n" % (1e3 * (time.perf_counter() - t0)))
        r = R.registration_icp(s2, t2, MAX_DIST, init, est, crit, comm=comm, shard=shard)
        # D2H: the RegistrationResult a Python user reads -- T, fitness, rmse AND the correspondence set (the
        # reference's pybind property copies it to the host, registration.cpp:338-343)
        cs = r.correspondence_set
        _ = (r.transformation, r.fitness, r.inlier_rmse)
        d2h[0] = C.sizeof(_lib.IcpResult) + cs.nbytes
        return r
    for _ in range(args.warmup):
        step_e2e()
    e2e_ms, res_e = timed(step_e2e, args.steps)
    h2d_bytes = h_src.nbytes + h_tgt.nbytes + h_tn.nbytes
    host_call_ms = None
    if not args.no_host_call:
        # the same end-to-end measurement through ONE C-ABI call that takes the host buffers itself
        # (cphb_registration_icp_host: uploads on a side stream, overlapped with the index build; the pairs come
        # back into a pinned host array)
        h_pairs = np.frombuffer((C.c_int32 * (2 * len(h_src))).from_address(L.cphb_malloc_host(8 * len(h_src))), dtype=np.int32).reshape(-1, 2)
        def step_host():
            return R.registration_icp_host(h_src, h_tgt, MAX_DIST, init, est, crit, target_normals=h_tn, comm=comm, shard=shard,
                                           return_correspondences=True, pairs_out=h_pairs)
        for _ in range(args.warmup):
            step_host()
        host_call_ms, res_h = timed(step_host, args.steps)
        assert np.array_equal(res_h.transformation, res_e.transformation), "host-buffer call and device call disagree"
        assert np.array_equal(res_h.correspondence_set, res_e.correspondence_set), "host-buffer call and device call disagree"

    # ---- kNN leg of the metric: SearchRadius(k=1, r) of the 1M source against the 1M target ------
    tree = cph.geometry.KDTreeFlann(t_pc)
    q_pc = cph.geometry.PointCloud(np.ascontiguousarray(src[lo:hi]))   # queries: no collective, shard by index
    for _ in range(2):
        tree.search_radius(q_pc.points, MAX_DIST, 1)
    knn_ms, _ = timed(lambda: tree.search_radius(q_pc.points, MAX_DIST, 1), args.steps)
    knn_steps = args.steps
    # ---- sub-records (N = 1 only; each a few device milliseconds) -----------------------------------
    extra = {}
    if world == 1 and not args.no_extras:
        # (a) the same registration with the certificates switched off (CPHB_CERT_GAIN=0): config 2 forces 30 iterations
        #     on a problem that converges in ~5, so `value` mostly measures launches whose searches are skipped by their
        #     certificates; this is the rate when every launch searches
        os.environ["CPHB_CERT_GAIN"] = "0"
        for _ in range(2):
            step_resident()
        nocert_ms, res_nc = timed(step_resident, args.steps)
        del os.environ["CPHB_CERT_GAIN"]
        assert np.array_equal(res_nc.transformation, res.transformation), "certificates changed the result"
        extra["certificates_off"] = {"value": ITERS * 1e3 / (nocert_ms / args.steps), "unit": "iter/s",
                                     "loop_iters_per_sec": ITERS * 1e3 / res_nc.loop_ms,
                                     "note": "same workload, every launch searches (CPHB_CERT_GAIN=0); identical result"}
        # (b) config 3 of BASELINE.json: VoxelDownSample(0.02) + SearchRadius(k=1, r=0.05) on 10 M points
        extra["config3"] = config3_records(cph, L, timed, peaks()[0], args)
    if not args.no_extras and args.points4 > 0:
        # (c) config 4 of BASELINE.json (the configuration it names for 8 GPUs) at EVERY N, so that the driver's 1 -> 8 runs
        #     time it: Generalized ICP 5 M -> 5 M, source sharded over the ranks
        c4 = config4_record(cph, L, timed, peaks()[0], args, rank, world, comm, dist)
        if rank == 0:
            extra["config4"] = c4
    if not args.no_extras and args.points5 > 0 and (world == 1 or args.config5_multi):
        # (d) config 5 of BASELINE.json: Colored-ICP pyramid on a 20 M-point pair.  In the default line at N = 1 only (the
        #     run that was validated on hardware this round); --config5-multi adds it at N > 1, where tools/bench_configs.py
        #     --config 5 is the maintained entry point (profiles/r1_n8_config5_n8.json)
        c5 = config5_record(cph, L, timed, args, rank, world, comm, dist)
        if rank == 0:
            extra["config5"] = c5
    if rank == 0:
        sampler.stop_flag = True
        sampler.join(timeout=2)

    # max over ranks
    if dist is not None:
        import torch
        t = torch.tensor([total_ms, e2e_ms, knn_ms, loop_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_ms, knn_ms, loop_ms = [float(x) for x in t.tolist()]
    if rank == 0:
        peak, peak_src = peaks()
        traffic = measured_traffic()
        ms_step = total_ms / args.steps
        value = ITERS * 1e3 / ms_step
        kern_ms = loop_ms / max(loop_launches, 1)
        # roofline: one "launch" = one fused iteration.  Its duration is the WHOLE launch loop (CUDA events around
        # it inside cphb_icp_run) divided by the number of iterations -- i.e. both instances of the iteration kernel
        # (search or certified pass; fixed-order sum + solve), a conservative (upper) figure for the kernel alone.
        n_fused = int(res.iterations) + 1
        fused_ms = loop_ms / max(n_fused, 1)
        units = (hi - lo)
        achieved = ALG_BYTES_PER_POINT * units / (fused_ms * 1e-3) / 1e9
        out = {
            "metric": "icp_iterations_per_sec", "value": value, "unit": "iter/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "points": n, "iterations": ITERS, "step": "one RegistrationICP call incl. index build",
                       "cache": "256 MiB memset between timed steps (L2 flush); working set ~60 MB",
                       "parallelism": "source sharded x%d (Hilbert-contiguous blocks), target replicated, 1 exchange(32 f64)/iter via %s"
                                      % (world, args.comm if world > 1 else "none")},
            "e2e": {"value": ITERS * 1e3 / (e2e_ms / args.steps), "unit": "iter/s", "h2d_bytes_per_step": int(h2d_bytes),
                    "d2h_bytes_per_step": int(d2h[0]), "ms_per_step": e2e_ms / args.steps},
            **({"e2e_host_call": {"value": ITERS * 1e3 / (host_call_ms / args.steps), "unit": "iter/s",
                                  "ms_per_step": host_call_ms / args.steps, "h2d_bytes_per_step": int(h2d_bytes),
                                  "call": "cphb_registration_icp_host"}} if host_call_ms else {}),
            "gpu_launches": int(launches),
            "loop": {"iters_per_sec": ITERS * 1e3 / loop_ms, "ms_per_launch": kern_ms, "launches": loop_launches,
                     "correspondences_per_sec": float(res.fitness) * n * (ITERS + 1) * 1e3 / loop_ms},
            "knn": {"mqueries_per_sec": n / (knn_ms / knn_steps) * 1e-3, "k": 1, "radius": MAX_DIST,
                    "ms": knn_ms / knn_steps,
                    "note": "SearchRadius of all %d source points (sharded by index over the ranks, no collective) incl. query ordering; aggregate rate" % n},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (traffic["traffic_bytes_per_launch"] if traffic and world == 1 and n == 1_000_000 else None),
                         "traffic_source": (traffic["source"] if traffic else None),
                         "peak_source": peak_src, "kernel": "icp_iteration_kernel<PointToPlane>",
                         "launch_ms": fused_ms, "launches": n_fused,
                         "launch_definition": "loop device time / iterations (both instances of the iteration kernel: search or certified pass, fixed-order sum, solve)",
                         "algorithmic_bytes_per_launch": ALG_BYTES_PER_POINT * units},
            "clocks": sampler.summary(),
            "step_ms": resident_steps_ms,
            "final": {"fitness": res.fitness, "inlier_rmse": res.inlier_rmse, "iterations": res.iterations,
                      "T": np.asarray(res.transformation).round(6).tolist()},
        }
        # headline e2e = the faster of the two public entry points (both move the same bytes: clouds in, result and
        # correspondence set out); both are printed
        if host_call_ms and host_call_ms < e2e_ms:
            out["e2e_device_api"] = dict(out["e2e"], call="PointCloud(host) + registration_icp + result.correspondence_set")
            out["e2e"] = {"value": ITERS * 1e3 / (host_call_ms / args.steps), "unit": "iter/s", "h2d_bytes_per_step": int(h2d_bytes),
                          "d2h_bytes_per_step": int(d2h[0]), "ms_per_step": host_call_ms / args.steps,
                          "call": "registration_icp_host (cphb_registration_icp_host: one C-ABI call on host buffers)"}
        else:
            out["e2e"]["call"] = "PointCloud(host) + registration_icp + result.correspondence_set"
        out.update(extra)
        if world == 1 and not args.no_cpu:
            out["cpu_baseline"], out["parity_vs_cpu_baseline"] = cpu_baseline(src, tgt, tn, res_e)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(out))
    for p in (p1, p2, p3):
        L.cphb_free_host(p)
    if comm is not None:
        barrier()
        L.cphb_comm_destroy(comm)
    if dist is not None:
        dist.destroy_process_group()


def cpu_baseline(src, tgt, tn, gpu_res):
    """Bounded CPU sample: up to 3 full 30-iteration registrations with the oracle port (kd-tree + OpenMP on all host
    cores), kd-tree build included -- the same unit of work as a GPU step -- median; plus the parity of the GPU result
    against this very run (BASELINE.md's "pose delta" and "index mismatches" columns)."""
    med, times, r, info = cpu_arm(src, tgt, tn, runs=3, budget_s=25.0)
    base = {"value": ITERS / med, "unit": "iter/s", "cores": info["threads"], "kind": "port",
            "sample": "%d full registrations: %d -> %d points, %d iterations, kd-tree build included; median %.2f s"
                      % (len(times), len(src), len(tgt), ITERS, med),
            **info, "final_fitness": r["fitness"], "final_rmse": r["inlier_rmse"]}
    a, b = gpu_res.correspondence_set, r["correspondence_set"]
    if a.shape == b.shape and np.array_equal(a, b):
        mism = 0
    else:
        ma, mb = np.full(len(src), -1, np.int64), np.full(len(src), -1, np.int64)
        ma[a[:, 0]] = a[:, 1]
        mb[b[:, 0]] = b[:, 1]
        mism = int((ma != mb).sum())
    parity = {"pose_delta_frobenius": float(np.linalg.norm(np.asarray(gpu_res.transformation, np.float64) - r["transformation"].astype(np.float64))),
              "index_mismatches": mism, "correspondences": int(len(b)),
              "fitness_delta": abs(float(gpu_res.fitness) - float(r["fitness"])),
              "rmse_delta": abs(float(gpu_res.inlier_rmse) - float(r["inlier_rmse"])),
              "tolerance": "pose <= 1e-5 Frobenius, indices bit-exact (north_star)"}
    return base, parity


def config4_record(cph, L, timed, peak, args, rank, world, comm, dist):
    """BASELINE.json config 4 as a sub-record at every N: Generalized ICP, 5 M -> 5 M points (analytic surface, normals
    given -> covariances), 30 iterations, r = 0.02, the source sharded over the ranks by the library (Hilbert-contiguous
    blocks), the target and its index replicated, one exchange of 32 float64 per iteration.  value = iterations / s of
    whole registrations (index build, source ordering, result included), clouds resident; max over ranks."""
    from cupoch_b200.testing import datagen
    R, G = cph.registration, cph.geometry
    n4 = args.points4
    tgt, tn = datagen.surface(n4, 11)
    src, sn = datagen.make_source(tgt, datagen.gt_transform(), 13, 14, 5e-4, attrs=[(tn, True)])
    t_pc, s_pc = G.PointCloud(tgt), G.PointCloud(src)
    t_pc.normals, s_pc.normals = tn, sn
    est, crit = R.TransformationEstimationForGeneralizedICP(1e-3), R.ICPConvergenceCriteria(0, 0, ITERS)
    s_c, t_c = R._with_covariances(s_pc, 1e-3), R._with_covariances(t_pc, 1e-3)
    shard = (rank, world) if world > 1 else None
    run = lambda: R.registration_icp(s_c, t_c, MAX_DIST, np.eye(4, dtype=np.float32), est, crit, comm=comm,
                                     return_correspondences=False, shard=shard)
    L.cphb_stream_synchronize(None)
    if dist is not None:
        dist.barrier()
    for _ in range(2):
        run()
    reps = 5
    steps, loops = [], []
    for _ in range(reps):   # one step at a time: per-step device times, max over ranks, then the median step
        m1, res = timed(run, 1)
        steps.append(m1)
        loops.append(res.loop_ms)
    if dist is not None:
        import torch
        t = torch.tensor([steps, loops], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        steps, loops = [float(x) for x in t[0].tolist()], [float(x) for x in t[1].tolist()]
    ms, loop_ms = float(np.median(steps)), float(np.median(loops))
    units = n4 // world
    launch_ms = loop_ms / (ITERS + 1)
    ach = 96 * units / (launch_ms * 1e-3) / 1e9
    gt = datagen.gt_transform()
    return {"workload": "config4: Generalized ICP %d -> %d, %d iters, r=%.2f, eps=1e-3, source sharded x%d" % (n4, n4, ITERS, MAX_DIST, world),
            "points": n4, "value": ITERS * 1e3 / ms, "unit": "iter/s", "ms_per_registration": ms,
            "step_ms": [round(x, 3) for x in steps], "aggregate": "median of %d steps (each the max over ranks)" % reps,
            "loop_iters_per_sec": ITERS * 1e3 / loop_ms, "scaling": "strong",
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "algorithmic_bytes_per_launch": 96 * units, "launch_ms": launch_ms,
                         "note": "per GPU: 96 B per source point of this rank's block (SURVEY 8d) / (loop time / 31 launches)"},
            "final": {"fitness": res.fitness, "inlier_rmse": res.inlier_rmse,
                      "pose_error_vs_ground_truth": float(np.linalg.norm(np.asarray(res.transformation, np.float64) - gt)),
                      "T": np.asarray(res.transformation).round(7).tolist()}}


def config5_record(cph, L, timed, args, rank, world, comm, dist):
    """BASELINE.json config 5 as a sub-record: Colored ICP 3-scale pyramid (voxel 0.05 / 0.025 / 0.0125, iterations
    50 / 30 / 14, relative criteria 1e-6 as in examples/python/advanced/colored_pointcloud_registration.py:37-60) on a
    20 M-point textured fragment pair over a 4 m x 4 m patch.  Per scale: VoxelDownSample -> EstimateNormals(radius 2v,
    30) -> colour gradient -> RegistrationColoredICP.  The pre-processing runs replicated on every rank (it needs no
    collective); the ICP loops shard the down-sampled source.  value = pyramids / s, end to end, clouds resident."""
    from cupoch_b200.testing import datagen
    R, G = cph.registration, cph.geometry
    n5 = args.points5
    tgt, _ = datagen.surface(n5, 31, extent=4.0)
    tc = datagen.texture(tgt, 32, 0.01)
    gt = datagen.gt_transform((0.0, 0.0, 2.0), (0.01, 0.0, 0.0))
    src, sc = datagen.make_source(tgt, gt, 33, 34, 2e-4, attrs=[(tc, False)])
    t_full, s_full = G.PointCloud(tgt), G.PointCloud(src)
    t_full.colors, s_full.colors = tc, sc
    shard = (rank, world) if world > 1 else None
    info = {}

    def pyramid():
        T = np.eye(4, dtype=np.float32)
        st = []
        for v, iters in ((0.05, 50), (0.025, 30), (0.0125, 14)):
            td, sd = t_full.voxel_down_sample(v), s_full.voxel_down_sample(v)
            td.estimate_normals(G.KDTreeSearchParamRadius(2 * v, 30))
            sd.estimate_normals(G.KDTreeSearchParamRadius(2 * v, 30))
            res = R.registration_colored_icp(sd, td, v, T, R.ICPConvergenceCriteria(1e-6, 1e-6, iters), comm=comm,
                                             return_correspondences=False, shard=shard)
            T = res.transformation
            st.append({"voxel": v, "n_src": len(sd), "n_tgt": len(td), "iterations": int(res.iterations), "fitness": res.fitness,
                       "rmse": res.inlier_rmse})
        info["stages"], info["T"] = st, T
        return T
    for _ in range(2):
        pyramid()
    reps = 3
    steps = []
    for _ in range(reps):
        m1, _ = timed(pyramid, 1)
        steps.append(m1)
    if dist is not None:
        import torch
        t = torch.tensor(steps, dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        steps = [float(x) for x in t.tolist()]
    ms = float(np.median(steps))
    return {"workload": "config5: Colored ICP 3-scale pyramid (0.05/0.025/0.0125; 50/30/14 iters) on a %d-point RGB fragment pair, "
                        "ICP loops sharded x%d, pre-processing replicated" % (n5, world),
            "points": n5, "value": 1e3 / ms, "unit": "pyramids/s", "ms_per_pyramid": ms, "step_ms": [round(x, 3) for x in steps],
            "aggregate": "median of %d steps (each the max over ranks)" % reps, "stages": info["stages"],
            "final": {"pose_error_vs_ground_truth": float(np.linalg.norm(np.asarray(info["T"], np.float64) - gt)),
                      "T": np.asarray(info["T"]).round(7).tolist()}}


def config3_records(cph, L, timed, peak, args):
    """BASELINE.json config 3 as sub-records with their own roofline (SURVEY 8d bytes): VoxelDownSample(0.02) of 10 M
    uniform points in [0,4)x[0,4)x[0,1), then SearchRadius(k=1, r=0.05) of the 10 M points against the down-sampled
    cloud.  Index build and query ordering are inside the timed search call, as in the reference's KDTreeFlann use."""
    from cupoch_b200.testing import datagen
    n3 = args.points3
    p = datagen.uniform_cube(n3, 21, hi=(4, 4, 1))
    pc = cph.geometry.PointCloud(p)
    for _ in range(2):
        down = pc.voxel_down_sample(0.02)
    reps = 5
    v_ms, down = timed(lambda: pc.voxel_down_sample(0.02), reps)
    v_ms /= reps
    n_out = len(down)
    v_bytes = 12 * n3 + 12 * n_out
    tree = cph.geometry.KDTreeFlann(down)
    for _ in range(2):
        tree.search_radius(pc.points, 0.05, 1)
    s_ms, out = timed(lambda: tree.search_radius(pc.points, 0.05, 1), reps)
    s_ms /= reps
    s_bytes = 32 * n3
    b_ms, _ = timed(lambda: cph.geometry.KDTreeFlann(down), reps)
    b_ms /= reps
    rec = lambda ms, by: {"achieved": by / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": by / (ms * 1e-3) / 1e9 / peak,
                          "bound": "hbm", "algorithmic_bytes": by}
    return {"workload": "config3: VoxelDownSample(0.02) + SearchRadius(k=1, r=0.05), %d points" % n3, "points": n3,
            "voxel": {"ms": v_ms, "mpoints_per_sec": n3 / v_ms * 1e-3, "n_out": int(n_out), "roofline": rec(v_ms, v_bytes)},
            "knn_10m": {"ms": s_ms, "mqueries_per_sec": n3 / s_ms * 1e-3, "found": int(out[0]), "targets": int(n_out),
                        "roofline": rec(s_ms, s_bytes), "index_build_ms": b_ms}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of each config-2 leg (the config 3/4/5 sub-records time fixed counts)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--e2e-host-call", action="store_true", help="(default now; kept for old command lines)")
    ap.add_argument("--no-host-call", action="store_true", help="skip the cphb_registration_icp_host e2e variant")
    ap.add_argument("--no-extras", action="store_true", help="skip the certificates-off and config-3 sub-records")
    ap.add_argument("--points3", type=int, default=10_000_000, help="size of the config-3 sub-records")
    ap.add_argument("--points4", type=int, default=5_000_000, help="size of the config-4 sub-record (0 = skip)")
    ap.add_argument("--points5", type=int, default=20_000_000, help="size of the config-5 sub-record (0 = skip)")
    ap.add_argument("--config5-multi", action="store_true", help="also run the config-5 sub-record at N > 1")
    ap.add_argument("--comm", default="p2p", choices=["p2p", "nccl"],
                    help="N>1 exchange: p2p = peer-memory stores fused into the reduce kernel, nccl = ncclAllReduce")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result of the last timed registration (transformation, fitness, inlier_rmse, "
                         "correspondence_set) as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_native(args, rank, world)


if __name__ == "__main__":
    main()
