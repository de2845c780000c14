#!/usr/bin/env python
"""bench.py — the headline measurement (BASELINE.json metric) for the filterpy hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one fused predict+update of a 2^20-filter bank, dim_x=4, dim_z=2, fp32, every
filter with its own F/H/Q/R (BASELINE.json configs[1]).  Weak scaling: every rank owns its own
2^20-filter bank (banks are independent, no data-path collective).  Prints ONE JSON line:

  value      filter-steps/s, whole job, inputs resident in HBM (CUDA events, max over ranks)
  e2e        same metric through the public API with HOST buffers: per step the measurement z is
             copied host->device from pinned memory and the posterior (x, P) device->host
  roofline   achieved HBM GB/s of the fused kernel vs MEASURED_PEAKS.json
  cpu_baseline  the oracle port (filterpy-shaped NumPy loop / vectorised NumPy / C) on host cores
  resample   systematic_resample of 2^26 particles (BASELINE.json configs[4], single-GPU slice)

`--impl reference` times the reference's CPU algorithm (the oracle port: the same per-filter
np.dot call sequence filterpy executes) on all host cores, bounded sample per step.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_FILTERS = 1 << 20
DIM_X, DIM_Z = 4, 2
BYTES_PER_FILTER_STEP = (2 * DIM_X + 4 * DIM_X * DIM_X + DIM_Z + DIM_Z * DIM_X + DIM_Z * DIM_Z) * 4  # 344
Z_RING = 4
DUMP_FILTERS = 1 << 19       # --dump-outputs: filters sampled from the bank (x and P of all 2^20 would be 80 MB)
METRIC = "kf_predict_update_filter_steps_per_sec"
UNIT = "filter-steps/s"
WORKLOAD = "kf_bank 2^20 filters dim_x=4 dim_z=2 fp32, per-filter F/H/Q/R, fused predict+update"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the fused kernel, from the committed
    `ncu --set full` capture (profiles/traffic.json); None when there is none."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["kf42_f32_kernel"]["dram_bytes_per_launch"]
    except Exception:
        return None


# ----------------------------------------------------------------------------- NUMA affinity
def pin_to_gpu_numa(local_rank):
    """Bind this process to the CPUs of the NUMA node its GPU hangs off (NVML PCI bus id ->
    /sys/bus/pci/devices/<id>/numa_node -> /sys/devices/system/node/node<k>/cpulist) BEFORE any pinned
    buffer is allocated: with several ranks per socket the host<->device copies of the e2e leg
    otherwise fight over the wrong memory controller.  Returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:                    # NVML: 00000000:1B:00.0, sysfs: 0000:1b:00.0
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return {"numa_node": None, "note": "no NUMA information for %s" % bus}
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus += list(range(int(lo), int(hi or lo) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as e:                                   # never fail the bench over affinity
        return {"numa_node": None, "note": "%s: %s" % (type(e).__name__, e)}


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    """SM clock and throttle reasons sampled from NVML while a region runs.  NVML is initialised
    when the object is built (outside any timed region); the thread polls every millisecond, so even
    a few-millisecond region is covered.  ``with sampler.region("name"):`` may be used several
    times; ``summary()`` reports the median over the device-timed steps and, when that region was
    too short to be caught, over the e2e steps (``sampled_in`` says which)."""

    def __init__(self, index):
        self.index = index
        self.samples = {}
        self.reasons = set()
        self.max_mhz = None
        self._h = None
        self._stop = threading.Event()
        self._th = None
        self._name = None
        try:
            import pynvml
            self._nv = pynvml
            pynvml.nvmlInit()
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
            self._names = {
                getattr(pynvml, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(pynvml, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(pynvml, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(pynvml, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            self._get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(pynvml, "nvmlDeviceGetCurrentClocksThrottleReasons")
        except Exception as e:  # no NVML: report nothing rather than guess
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def _sample(self):
        self.samples.setdefault(self._name, []).append(self._nv.nvmlDeviceGetClockInfo(self._h, self._nv.NVML_CLOCK_SM))
        r = self._get_reasons(self._h)
        for bit, nm in self._names.items():
            if r & bit:
                self.reasons.add(nm)

    def _run(self):
        try:
            while not self._stop.is_set():
                self._sample()
                time.sleep(0.001)
        except Exception as e:
            self.reasons.add("nvml_error:%s" % type(e).__name__)

    def region(self, name):
        self._name = name
        return self

    def __enter__(self):
        if self._h is not None:
            self._stop.clear()
            self._th = threading.Thread(target=self._run, daemon=True)
            self._th.start()
        return self

    def __exit__(self, *a):
        if self._th is not None:
            self._stop.set()
            self._th.join(timeout=2)
            self._th = None

    def summary(self):
        for name in ("device_timed_steps", "e2e_steps"):
            if self.samples.get(name):
                return {"sm_mhz": float(np.median(self.samples[name])), "sm_max_mhz": self.max_mhz,
                        "reasons": sorted(self.reasons), "sampled_in": name, "n_samples": len(self.samples[name])}
        return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ----------------------------------------------------------------------------- CPU legs
def reference_importable():
    """The unmodified reference (filterpy 1.4.5) when __graft_entry__.build() installed a copy under
    oracle/_ref (oracle/reference.py).  Returns the sys.path entry or None."""
    from oracle import reference
    return reference.importable()


def _loop_port_worker(args):
    """One worker = one host core.  kind "reference": real filterpy.kalman.KalmanFilter objects,
    predict(); update(z) in a Python loop — the reference as shipped.  kind "port": the oracle's
    per-filter functions with the reference's np.dot call sequence (oracle.kf.*_single ==
    kalman_filter.py:471-478, 533-556)."""
    seed, nf, steps, ref_path, core = args
    try:
        os.sched_setaffinity(0, {core})                     # one worker per core, BLAS threads off (set before the fork)
    except Exception:
        pass
    from filterpy_b200.common import workloads as wl
    w = wl.kf_bank_cv2d(nf, seed=seed, steps=steps)
    if ref_path is not None:
        if ref_path not in sys.path:
            sys.path.insert(0, ref_path)
        from filterpy.kalman import KalmanFilter as RefKF
        kfs = []
        for i in range(nf):
            f = RefKF(dim_x=DIM_X, dim_z=DIM_Z)
            f.x = w["x"][i].copy(); f.P = w["P"][i].copy(); f.F = w["F"][i]; f.H = w["H"][i]; f.Q = w["Q"][i]; f.R = w["R"][i]
            kfs.append(f)
        t0 = time.perf_counter()
        for t in range(steps):
            zt = w["zs"][t]
            for i in range(nf):
                kfs[i].predict(); kfs[i].update(zt[i])
        return time.perf_counter() - t0
    from oracle import kf as okf
    xs = [w["x"][i] for i in range(nf)]; Ps = [w["P"][i] for i in range(nf)]
    t0 = time.perf_counter()
    for t in range(steps):
        for i in range(nf):
            x, P = okf.kf_predict_single(xs[i], Ps[i], w["F"][i], w["Q"][i])
            xs[i], Ps[i] = okf.kf_update_single(x, P, w["zs"][t, i], w["H"][i], w["R"][i])[:2]
    return time.perf_counter() - t0


def cpu_loop_port(cores, nf_per_core, steps, ref_path=None):
    """Returns (filter-steps/s, wall seconds, per-worker seconds)."""
    import multiprocessing as mp
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[v] = "1"                                 # inherited by the forked workers: no BLAS thread pools fighting
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)
    except Exception:
        pass
    avail = sorted(os.sched_getaffinity(0))
    cores = min(cores, len(avail))
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        t0 = time.perf_counter()
        times = pool.map(_loop_port_worker, [(100 + i, nf_per_core, steps, ref_path, avail[i]) for i in range(cores)])
        wall = time.perf_counter() - t0
    # throughput of `cores` workers running concurrently: each timed its own loop (input generation
    # and process start-up excluded); the slowest worker bounds the step
    return cores * nf_per_core * steps / max(times), wall, times


def cpu_vectorised_port(nf, steps):
    from oracle import kf as okf
    from filterpy_b200.common import workloads as wl
    w = wl.kf_bank_cv2d(nf, seed=1, steps=1)
    x, P = w["x"], w["P"]
    t0 = time.perf_counter()
    for _ in range(steps):
        o = okf.kf_step_bank(x, P, w["zs"][0], w["F"], w["H"], w["Q"], w["R"]); x, P = o["x"], o["P"]
    wall = time.perf_counter() - t0
    return nf * steps / wall, wall


def cpu_c_port(nf, steps, threads):
    import ctypes
    from concurrent.futures import ThreadPoolExecutor
    from oracle import cbuild
    from filterpy_b200.common import workloads as wl
    lib = cbuild.load()
    w = wl.kf_bank_cv2d(nf, seed=2, steps=1)
    x, P = w["x"].copy(), w["P"].copy()
    z = np.ascontiguousarray(w["zs"][0])
    chunk = (nf + threads - 1) // threads

    def run(i):
        a, b = i * chunk, min(nf, (i + 1) * chunk)
        if a >= b:
            return 0
        p = lambda arr, off: ctypes.c_void_p(arr.ctypes.data + off * arr.itemsize)
        return lib.oracle_kf_step_f64(ctypes.c_int64(b - a), 4, 2, p(x, a * 4), p(P, a * 16),
                                      p(w["F"], a * 16), ctypes.c_int64(16), p(w["H"], a * 8), ctypes.c_int64(8),
                                      p(w["Q"], a * 16), ctypes.c_int64(16), p(w["R"], a * 4), ctypes.c_int64(4),
                                      p(z, a * 2), None, ctypes.c_double(1.0), 1)
    with ThreadPoolExecutor(threads) as ex:
        t0 = time.perf_counter()
        for _ in range(steps):
            list(ex.map(run, range(threads)))
        wall = time.perf_counter() - t0
    return nf * steps / wall, wall


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port) on all host cores."""
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) or 1
    nf_per_core = 2048          # bounded sample of the 2^20-filter bank per step
    ref_path = reference_importable()
    kind = "reference" if ref_path else "port"
    for _ in range(min(args.warmup, 1)):
        cpu_loop_port(cores, 256, 1, ref_path)
    val, wall, times = cpu_loop_port(cores, nf_per_core, args.steps, ref_path)
    sample = "%d filters/core x %d cores x %d steps of the 2^20 bank (%s), one pinned worker per core, BLAS threads = 1, worker seconds min/median/max %.2f/%.2f/%.2f" % (
        nf_per_core, cores, args.steps,
        "real filterpy.kalman.KalmanFilter objects from %s" % ref_path if ref_path else "filterpy-shaped NumPy loop, oracle port",
        min(times), float(np.median(times)), max(times))
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU legs
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from filterpy_b200.kalman import KalmanFilter
    from filterpy_b200.common import workloads as wl

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    all_cpus = os.sched_getaffinity(0)
    affinity = pin_to_gpu_numa(local_rank) if not args.no_pin else {"numa_node": None, "note": "disabled"}
    K, W = args.steps, max(args.warmup, 3)
    N = N_FILTERS

    w = wl.kf_bank_cv2d(N, seed=1234 + rank, steps=Z_RING, dtype=np.float32)
    kf = KalmanFilter(DIM_X, DIM_Z, n_filters=N, dtype=np.float32, device=dev, diagnostics=False)
    for k in "xPFHQR":
        setattr(kf, k, w[k])
    z_dev = [torch.from_numpy(w["zs"][i]).to(dev) for i in range(Z_RING)]
    z_pin = [torch.from_numpy(w["zs"][i]).pin_memory() for i in range(Z_RING)]
    x_pin = torch.empty((N, DIM_X), dtype=torch.float32).pin_memory()
    P_pin = torch.empty((N, DIM_X, DIM_X), dtype=torch.float32).pin_memory()
    x0, P0 = kf.x.clone(), kf.P.clone()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def reset():
        # in place: the captured graph and the cached launch arguments hold the addresses of x and P,
        # so every timed step, replayed or direct, advances the state a caller reads
        kf.x.copy_(x0); kf.P.copy_(P0)

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # ---- value: inputs resident in HBM -----------------------------------------------------
    # The K steps are issued as CUDA-graph replays of Z_RING consecutive steps (one fused kernel per
    # step, the ring's measurement buffers in turn); a remainder of K % Z_RING steps is launched
    # directly.  Same kernels, same work; the graph only removes per-launch host latency.
    def step_resident(i):
        kf.predict()
        kf.update(z_dev[i % Z_RING])

    def ring():
        for i in range(Z_RING):
            step_resident(i)

    clk = ClockSampler(local_rank)            # NVML is initialised here, outside every timed region
    use_graph = not args.no_graph
    graph = kf.capture(ring) if use_graph else None
    reset()
    for i in range(W):
        step_resident(i)
    if graph is not None:
        graph.replay()
    barrier()
    reps, rem = (K // Z_RING, K % Z_RING) if graph is not None else (0, K)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + rem + 1)]
    with clk.region("device_timed_steps"):
        evs[0].record()
        for r in range(reps):
            graph.replay()
            evs[r + 1].record()
        for i in range(rem):
            step_resident(i)
            evs[reps + i + 1].record()
        barrier()
    total_ms = max_over_ranks(evs[0].elapsed_time(evs[reps + rem]))
    per_launch_ms = np.array([evs[r].elapsed_time(evs[r + 1]) / Z_RING for r in range(reps)] +
                             [evs[reps + i].elapsed_time(evs[reps + i + 1]) for i in range(rem)])
    value = world * N * K / (total_ms * 1e-3)
    dump = None
    if args.dump_outputs and rank == 0:
        # the posterior of the last timed step, for a fixed sample of the filters
        sel = torch.from_numpy(np.sort(np.random.default_rng(0).choice(N, DUMP_FILTERS, replace=False))).to(dev)
        dump = {"x": kf.x.index_select(0, sel).cpu().numpy(), "P": kf.P.index_select(0, sel).cpu().numpy()}

    # ---- e2e: host buffers, copies inside the timed region -----------------------------------
    # Every step copies that step's measurements from pinned host memory to the device
    # (kf.update is handed the HOST tensor), runs the fused step, and copies the posterior back to
    # pinned host memory.  Primary figure: the posterior mean x (what a tracker reads every epoch);
    # `e2e_full_posterior` also brings P back (92 MB/step: PCIe-bound).  The device->host copies
    # run on a side stream from a snapshot of the state, so they overlap the next step's H2D copy
    # and kernel (PCIe is full duplex); the timed region ends when every copy has landed.
    copy_stream = torch.cuda.Stream(dev)
    snap_x = [torch.empty_like(x0) for _ in range(2)]
    snap_P = [torch.empty_like(P0) for _ in range(2)]
    snap_free = [torch.cuda.Event() for _ in range(2)]

    def step_e2e(i, with_P):
        kf.predict()
        kf.update(z_pin[i % Z_RING])                   # H2D of this step's measurements + fused kernel
        b = i & 1
        cur = torch.cuda.current_stream(dev)
        cur.wait_event(snap_free[b])                   # the D2H that last used this snapshot is done
        snap_x[b].copy_(kf.x)
        if with_P:
            snap_P[b].copy_(kf.P)
        ready = torch.cuda.Event()
        ready.record(cur)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ready)
            x_pin.copy_(snap_x[b], non_blocking=True)  # D2H of the posterior
            if with_P:
                P_pin.copy_(snap_P[b], non_blocking=True)
            snap_free[b].record(copy_stream)

    def run_e2e(with_P):
        reset()
        for i in range(W):
            step_e2e(i, with_P)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with clk.region("e2e_steps"):
            e0.record()
            for i in range(K):
                step_e2e(i, with_P)
            torch.cuda.current_stream(dev).wait_stream(copy_stream)
            e1.record()
            barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    e2e_ms = run_e2e(False)
    e2e_value = world * N * K / (e2e_ms * 1e-3)
    e2e_full_ms = run_e2e(True)
    h2d = N * DIM_Z * 4
    d2h = N * DIM_X * 4
    d2h_full = N * (DIM_X + DIM_X * DIM_X) * 4

    # ---- the other BASELINE configurations, weak-scaled like C2 (every rank its own bank), and the
    # particle path: the GLOBAL 2^26-particle set sharded over the ranks
    peak, peak_src = peaks()
    extras = {}
    if not args.no_extra:
        kf = None; graph = None                             # free the C2 bank before the next ones are built
        torch.cuda.empty_cache()
        extras = extra_legs(dev, rank, world, peak, max_over_ranks, barrier)
    res = None
    if not args.no_resample:
        res = resample_leg(dev, args, rank, world, peak, max_over_ranks, barrier)
    if rank != 0:
        return
    kern_ms = float(np.mean(per_launch_ms))
    achieved = BYTES_PER_FILTER_STEP * N / (kern_ms * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "filters_per_gpu": N, "parallelism": "bank sharded, %d rank(s)" % world,
                   "l2": "inputs larger than L2 (344 MB touched per step vs 126 MB L2)",
                   "launch": ("CUDA graph of %d steps per replay" % Z_RING) if use_graph else "one launch per step"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / K, "result": "posterior mean x[N,4] per step"},
        "e2e_full_posterior": {"value": world * N * K / (e2e_full_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                               "d2h_bytes_per_step": d2h_full, "ms_per_step": e2e_full_ms / K,
                               "result": "posterior x[N,4] and P[N,4,4] per step"},
        "gpu_launches": K,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": ncu_traffic(), "peak_source": peak_src,
                     "kernel": "kf42_f32_kernel<3,false,false>", "bytes_per_launch": BYTES_PER_FILTER_STEP * N,
                     "kernel_ms": kern_ms, "kernel_ms_min": float(per_launch_ms.min())},
        "clocks": clk.summary(),
        "affinity": affinity,
    }
    line.update(extras)
    if res is not None:
        line["resample"] = res
    if world == 1 and not args.no_cpu:
        try:
            os.sched_setaffinity(0, all_cpus)               # the CPU legs use every host core again
        except Exception:
            pass
        cores = os.cpu_count() or 1
        cores = len(os.sched_getaffinity(0)) or cores
        ref_path = reference_importable()
        lp, lp_wall, _ = cpu_loop_port(cores, 1024, 2, ref_path)
        vp, vp_wall = cpu_vectorised_port(1 << 17, 3)
        cp, cp_wall = cpu_c_port(1 << 19, 4, cores)
        line["cpu_baseline"] = {
            "value": lp, "unit": UNIT, "cores": cores, "kind": "reference" if ref_path else "port",
            "sample": "%s, %d filters/core x %d pinned cores x 2 steps, BLAS threads = 1, %.1f s"
                      % ("real filterpy.kalman.KalmanFilter objects" if ref_path else "filterpy-shaped NumPy loop (oracle.kf.*_single)",
                         1024, cores, lp_wall),
            "vectorised_numpy": {"value": vp, "cores": 1, "sample": "2^17 filters x 3 steps, %.1f s" % vp_wall},
            "c_port": {"value": cp, "cores": cores, "sample": "2^19 filters x 4 steps fp64, %.1f s" % cp_wall},
        }
    print(json.dumps(line), flush=True)
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)


def timed_steps(fn, reps, warm, dev, max_over_ranks, barrier):
    """mean device time (ms) of one call of fn: CUDA events around `reps` calls, max over ranks"""
    import torch
    for _ in range(warm):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    barrier()
    return max_over_ranks(e0.elapsed_time(e1)) / reps


def extra_legs(dev, rank, world, peak, max_over_ranks, barrier):
    """BASELINE configs 3 and 4 and the drop-in default of config 2 (diagnostics=True: K, S, SI, y,
    priors, log-likelihood written every step), each with the roofline of its kernel; weak scaling."""
    import torch
    from filterpy_b200.kalman import (KalmanFilter, UnscentedKalmanFilter, MerweScaledSigmaPoints, ConstVelFx, RangeAzElHx)
    from filterpy_b200.common import workloads as wl
    out = {}

    def roof(ms, units, bpu, kernel):
        gbs = units * bpu / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                "bytes_per_launch": units * bpu, "kernel_ms": ms, "kernel": kernel}

    # C2 with the optional outputs (what a filterpy object exposes after every update)
    N = N_FILTERS
    w = wl.kf_bank_cv2d(N, seed=1234 + rank, steps=1, dtype=np.float32)
    kf = KalmanFilter(DIM_X, DIM_Z, n_filters=N, dtype=np.float32, device=dev, diagnostics=True)
    for k in "xPFHQR":
        setattr(kf, k, w[k])
    z = torch.from_numpy(w["zs"][0]).to(dev)

    def step2():
        kf.predict(); kf.update(z)
    ms = timed_steps(step2, 20, 3, dev, max_over_ranks, barrier)
    extra_b = (DIM_X + DIM_X * DIM_X + DIM_X * DIM_Z + DIM_Z + 2 * DIM_Z * DIM_Z + 1) * 4 + 4      # priors, K, y, S, SI, loglik, status
    out["kf_c2_diagnostics"] = {"workload": "config 2 with diagnostics=True (x_prior, P_prior, K, y, S, SI, log-likelihood, status written)",
                                "value": world * N / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "dtype": "f32",
                                "roofline": roof(ms, N, BYTES_PER_FILTER_STEP + extra_b, "kf42_f32_kernel<3,false,true>")}
    del kf, z, w
    torch.cuda.empty_cache()

    # C3: 10 M filters 9/3 fp64 over 8 GPUs = 1.25 M per rank
    N3 = 1250000
    small = wl.kf_bank_ca3d(50000, seed=4321 + rank, steps=1)
    w3 = {k: np.concatenate([v] * 25, axis=1 if k == "zs" else 0) for k, v in small.items()}
    kf3 = KalmanFilter(9, 3, n_filters=N3, dtype=np.float64, device=dev, diagnostics=False)
    for k in "xPFHQR":
        setattr(kf3, k, w3[k])
    z3 = torch.from_numpy(w3["zs"][0]).to(dev)

    def step3():
        kf3.predict(); kf3.update(z3)
    ms = timed_steps(step3, 10, 3, dev, max_over_ranks, barrier)
    bpu3 = (2 * 9 + 4 * 81 + 3 + 27 + 9) * 8
    out["kf_c3"] = {"workload": "config 3: 9/3 fp64, per-filter F/H/Q/R, 1.25 M filters per GPU (10 M over 8)",
                    "filters_per_gpu": N3, "value": world * N3 / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "dtype": "f64",
                    "roofline": roof(ms, N3, bpu3, "kf_rowblock_kernel<double,9,3>")}
    # C3 the drop-in way (diagnostics=True): the optional outputs are staged in shared memory and leave with bulk stores
    kf3d = KalmanFilter(9, 3, n_filters=N3, dtype=np.float64, device=dev, diagnostics=True)
    for k in "xPFHQR":
        setattr(kf3d, k, w3[k])

    def step3d():
        kf3d.predict(); kf3d.update(z3)
    ms = timed_steps(step3d, 10, 3, dev, max_over_ranks, barrier)
    extra3 = (9 + 81 + 27 + 3 + 2 * 9 + 1) * 8 + 4            # priors, K, y, S, SI, loglik, status
    out["kf_c3_diagnostics"] = {"workload": "config 3 with diagnostics=True (x_prior, P_prior, K, y, S, SI, log-likelihood, status written)",
                                "filters_per_gpu": N3, "value": world * N3 / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "dtype": "f64",
                                "roofline": roof(ms, N3, bpu3 + extra3, "kf_rowblock_kernel<double,9,3,EXTRAS>")}
    del kf3, kf3d, z3, w3, small
    torch.cuda.empty_cache()

    # batch_filter (BASELINE configs[0]'s call, as a bank): 2^18 filters x 32 epochs inside ONE kernel, 4/2 fp32
    Nb, Tb = 1 << 18, 32
    wb = wl.kf_bank_cv2d(Nb, seed=99 + rank, steps=Tb, dtype=np.float32)
    kfb = KalmanFilter(DIM_X, DIM_Z, n_filters=Nb, dtype=np.float32, device=dev, diagnostics=False)
    for k in "xPFHQR":
        setattr(kfb, k, wb[k])
    zsb = torch.from_numpy(wb["zs"]).to(dev)
    ms = timed_steps(lambda: kfb.batch_filter(zsb), 5, 3, dev, max_over_ranks, barrier)
    bpub = (DIM_Z + 2 * DIM_X + 2 * DIM_X * DIM_X) * 4          # z in; means, covariances, means_p, covariances_p out
    out["kf_batch_filter"] = {"workload": "KalmanFilter.batch_filter, 2^18 filters x 32 epochs per call and GPU, 4/2 fp32, time loop in the kernel",
                              "filters_per_gpu": Nb, "epochs": Tb, "value": world * Nb * Tb / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
                              "dtype": "f32", "roofline": roof(ms, Nb * Tb, bpub, "kf_batch_kernel<float,4,2,staged>")}
    del kfb, zsb, wb
    torch.cuda.empty_cache()

    # C4: UKF Merwe 6/3, 2^18 filters, CV + range/azimuth/elevation, fp64
    N4 = 1 << 18
    uw = wl.ukf_bank_cv3d(N4, seed=2468 + rank, steps=1)
    u = UnscentedKalmanFilter(6, 3, 0.1, RangeAzElHx(), ConstVelFx(), MerweScaledSigmaPoints(6, .5, 2., 0.),
                              n_filters=N4, dtype=np.float64, device=dev, diagnostics=False)
    u.x = uw["x"]; u.P = uw["P"]; u.Q = uw["Q"]; u.R = uw["R"]
    z4 = torch.from_numpy(uw["zs"][0]).to(dev)

    def step4():
        u.predict(); u.update(z4)
    ms = timed_steps(step4, 20, 3, dev, max_over_ranks, barrier)
    bpu4 = (2 * 6 + 3 * 36 + 3 + 9) * 8
    out["ukf_c4"] = {"workload": "config 4: UKF MerweScaledSigmaPoints(6, .5, 2, 0), CV + range/azimuth/elevation, 2^18 filters per GPU",
                     "filters_per_gpu": N4, "value": world * N4 / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "dtype": "f64",
                     "roofline": roof(ms, N4, bpu4, "ukf_kernel<double,6,3,CV,RangeAzEl>")}
    del u, z4, uw
    torch.cuda.empty_cache()

    # the tensor-core tile (DESIGN.md §3.2c): predict of shared-model fp32 banks with dim_x = 16 / 32 on tcgen05.mma
    # (three-term TF32 split); algorithmic bytes per filter: x and P in, x and P out
    for n_tc, N_tc in ((16, 1 << 19), (32, 1 << 17)):
        rng = np.random.default_rng(77 + rank)
        a = rng.normal(size=(2048, n_tc, n_tc)).astype(np.float32)
        P0 = np.tile(2.0 * (a @ np.swapaxes(a, -1, -2) / n_tc + np.eye(n_tc, dtype=np.float32)), (N_tc // 2048, 1, 1))
        kt = KalmanFilter(n_tc, 4, n_filters=N_tc, dtype=np.float32, device=dev, diagnostics=False)
        kt.x, kt.P = np.tile(rng.normal(size=(2048, n_tc)).astype(np.float32), (N_tc // 2048, 1)), P0
        kt.F, kt.H = np.eye(n_tc) + 0.05 * rng.normal(size=(n_tc, n_tc)), rng.normal(size=(4, n_tc))
        kt.Q, kt.R = 0.05 * np.eye(n_tc), 0.5 * np.eye(4)

        def step_tc():
            kt.predict(); kt._flush()
        ms = timed_steps(step_tc, 20, 3, dev, max_over_ranks, barrier)
        out["kf_tc_predict_%d" % n_tc] = {
            "workload": "KalmanFilter.predict of a shared-model fp32 bank, dim_x = %d, %d filters per GPU, on tcgen05.mma (kind::tf32, 3-term split)" % (n_tc, N_tc),
            "filters_per_gpu": N_tc, "value": world * N_tc / (ms * 1e-3), "unit": "filter-predicts/s", "ms_per_step": ms, "dtype": "f32 (tf32x3 products, f32 accumulate)",
            "roofline": roof(ms, N_tc, (2 * n_tc + 2 * n_tc * n_tc) * 4, "kf_cov_tc_kernel<%d,0>" % n_tc)}
        # the whole step in the tile: H and R shared too, dim_z = 4 (P' H' as a third tensor-core product, the dim_z-sized
        # pieces per filter on the CUDA cores); algorithmic bytes: x, P, z in; x, P out
        z_tc = torch.from_numpy(rng.normal(size=(N_tc, 4)).astype(np.float32)).to(dev)

        def step_tc_fused():
            kt.predict(); kt.update(z_tc)
        ms = timed_steps(step_tc_fused, 20, 3, dev, max_over_ranks, barrier)
        out["kf_tc_step_%d" % n_tc] = {
            "workload": "KalmanFilter.predict + update of a shared-model fp32 bank, %d/4, %d filters per GPU, one launch on tcgen05.mma (kind::tf32, 3-term split)" % (n_tc, N_tc),
            "filters_per_gpu": N_tc, "value": world * N_tc / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "dtype": "f32 (tf32x3 products, f32 accumulate)",
            "roofline": roof(ms, N_tc, (2 * n_tc + 2 * n_tc * n_tc + 4) * 4, "kf_cov_tc_kernel<%d,4>" % n_tc)}
        del kt, P0, a, z_tc
        torch.cuda.empty_cache()
    return out


def resample_leg(dev, args, rank, world, peak, max_over_ranks, barrier):
    """BASELINE configs[4]: systematic_resample of the GLOBAL 2^26-particle set.  One GPU: the
    single-array call.  N GPUs: the weights sharded contiguously, one all-gather of the shard sums
    and one of the shard composites (NCCL), every rank emits its span of the output
    (filterpy_b200.distributed.sharded_systematic_resample); particles/s = 2^26 / max-rank time.
    The result is checked against the C oracle (every rank its own span) once, outside the timing."""
    import torch
    import torch.distributed as dist
    from filterpy_b200.monte_carlo import resampling as rs
    from filterpy_b200 import distributed as bd
    from filterpy_b200.common import workloads as wl
    N = 1 << 26
    wts = wl.resample_weights(N, "heavy", seed=97)
    np.random.seed(7)
    u = float(np.random.random())
    reps = 10
    info = None
    if world == 1:
        wd = torch.from_numpy(wts).to(dev)
        plan = rs.ResamplePlan(N, device=dev)
        ms = timed_steps(lambda: plan.systematic(wd, u), reps, 3, dev, max_over_ranks, barrier)
        got, lo = plan.indexes, 0
        info = plan.info().tolist()
        exchange = "none (single array)"
        # stratified at the same size (resampling.py:80-114; 20 B/particle: the uniforms are read too)
        U = torch.from_numpy(np.random.default_rng(5).random(N)).to(dev)
        ms_str = timed_steps(lambda: plan.stratified(wd, U), 5, 2, dev, max_over_ranks, barrier)
        plan.systematic(wd, u)
    else:
        b = bd.shard_bounds(N, world)
        sizes = [int(b[r + 1] - b[r]) for r in range(world)]
        w_loc = torch.from_numpy(wts[int(b[rank]):int(b[rank + 1])]).to(dev)
        splan = bd.ShardedResamplePlan(sizes, device=dev)
        ms = timed_steps(lambda: splan.resample(w_loc, u), reps, 3, dev, max_over_ranks, barrier)
        lo, hi = [int(v) for v in splan.out_range.cpu().numpy()]
        got = splan.indexes[:hi - lo]
        info = splan.info.cpu().numpy().tolist() + [int(splan.status.item())]
        exchange = "all-gather of %d shard sums + all-gather of %d shard composites (NCCL), no serial hand-over" % (world, world)
        ms_str = None
    t = ms * 1e-3
    out = {"metric": "systematic_resample_particles_per_sec", "particles": N, "n_gpus": world, "value": N / t, "unit": "particles/s",
           "ms": ms, "exchange": exchange,
           "roofline": {"bound": "hbm", "achieved": 12.0 * N / world / t / 1e9, "peak": peak, "unit": "GB/s per GPU",
                        "frac": 12.0 * N / world / t / 1e9 / peak, "bytes_per_particle": 12},
           "info": info}
    if ms_str is not None:
        out["stratified"] = {"ms": ms_str, "value": N / (ms_str * 1e-3), "unit": "particles/s",
                             "roofline_frac": 20.0 * N / (ms_str * 1e-3) / 1e9 / peak, "bytes_per_particle": 20}
    if not args.no_cpu:
        # bit-exactness against the oracle, and the CPU baseline (rank 0 times it)
        from oracle import resample as ors
        t0 = time.perf_counter()
        want = ors.systematic_resample_c(wts, u)
        tc = time.perf_counter() - t0
        mine = got.cpu().numpy()
        ok = bool(np.array_equal(mine, want[lo:lo + len(mine)]))
        if world > 1:
            flag = torch.tensor([1 if ok else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok = bool(flag.item())
            cover = torch.tensor([len(mine)], device=dev, dtype=torch.int64)
            dist.all_reduce(cover)
            ok = ok and int(cover.item()) == N
        out["bit_exact_vs_oracle"] = ok
        out["cpu_baseline"] = {"value": N / tc, "unit": "particles/s", "cores": 1, "kind": "port",
                               "sample": "oracle.c sequential cumsum + merge on all 2^26 particles, %.2f s" % tc}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-resample", action="store_true", help="skip the resample leg")
    ap.add_argument("--no-graph", action="store_true", help="launch every step directly instead of CUDA-graph replays")
    ap.add_argument("--no-pin", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--no-extra", action="store_true", help="skip the C2-diagnostics / C3 / C4 legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the posterior of the last one as DIR/x.npy (N,4) and "
                         "DIR/P.npy (N,4,4), fp32, for a fixed seeded sample of 2^19 of rank 0's filters")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
