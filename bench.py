"""
bench.py -- anomaly windows/sec of the fused predict+score hot path on BASELINE.json configs[1]:
1 000 machines x 64-tag feedforward_hourglass autoencoder, 10 000 rows per machine, per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--machines M] [--rows R] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path (gb_ffae_infer_score) over every machine of the rank: 10^7 windows per GPU, inputs
resident in HBM.  `value` is whole-job windows/s (all ranks' windows / max-over-ranks device time).  `e2e` repeats the
measurement through the fleet API with HOST buffers: pinned H2D of x and y and D2H of every output inside the timed
region.  `roofline` is the algorithmic HBM bytes (1 548 B/window, SURVEY 8d) over the CUDA-event time, against the
measured copy bandwidth in MEASURED_PEAKS.json.  `cpu_baseline` times the CPU oracle (a restatement of the reference's
Keras predict loop + diff.py arithmetic -- NOT TensorFlow, which is not installable here, and not the reference's own diff.py,
which lives under /root/reference and does not exist on the GPU box) on a bounded sample, imports warmed, arithmetic only.
Machines shard across ranks with no data-path collective (weak scaling: the per-GPU workload is fixed); NCCL only
broadcasts the machine assignment and gathers one score summary per machine after the timed region.  Beside the weak-scaling
`value` the line carries `strong` (the SAME 1 000 machines split over the N ranks, BASELINE's "1k machines at 1/2/4/8 B200") and
`secondary` (one GPU's share of BASELINE configs[2], [3] and the configs[4] request shape, benchmarks/secondary.py, ~20 s).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T = 64
BYTES_PER_WINDOW = 4 * T + 4 * T + 4 * 4 * T + 12  # read x, y; write model-output, 2 tag-anomaly blocks, confidence; 3 row scalars
# dram__bytes_read.sum + dram__bytes_write.sum per window from the committed `ncu --set full` captures (profiles/, file names below)
NCU_DRAM_BYTES_PER_WINDOW = {"tcgen05": (1.569383e9 + 3.048933e9) / 3.0e6, "fma": (1.037003e9 + 2.019607e9) / 2.0e6}
NCU_SOURCE = {"tcgen05": "profiles/r02_ffae_tc_ncu.txt (300-machine capture)", "fma": "profiles/r01_ffae_infer_fma_ncu.txt (200-machine capture)"}
DUMP_BYTES = 32 << 20  # --dump-outputs: a seeded sample of rows of every output, this many bytes in all
METRIC = "anomaly windows/sec (64-tag feedforward_hourglass AE, 1k machines x 10k rows per GPU, fused predict+score)"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def host_info():
    """What the CPU numbers were measured on: usable cores (affinity AND cgroup quota), load, NUMA layout."""
    cores = len(os.sched_getaffinity(0))
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, period = f.read().split()
            quota = None if q == "max" else float(q) / float(period)
    except Exception:
        pass
    try:
        load = os.getloadavg()
    except Exception:
        load = None
    usable = cores if quota is None else max(1, min(cores, int(quota)))
    return {"affinity_cores": cores, "cgroup_cpu_max": quota, "usable_cores": usable, "loadavg": load}


def bind_to_gpu_numa_node(local_rank: int):
    """
    Pin this rank's threads to the CPUs of its GPU's NUMA node BEFORE any pinned host memory is allocated (first touch then puts the
    staging buffers on that node): the end-to-end path moves 15.5 GB per step per GPU through host DRAM, and with eight ranks an
    unbound process streams half of it across the socket interconnect.  Returns a description for the JSON line.
    """
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=index,pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout
        bus = {int(l.split(",")[0]): l.split(",")[1].strip() for l in out.strip().splitlines()}[local_rank]
        dom, rest = bus.split(":", 1)
        sysfs = f"/sys/bus/pci/devices/{dom[-4:].lower()}:{rest.lower()}/numa_node"
        node = int(open(sysfs).read())
        if node < 0:
            return {"numa_node": None, "bound": False, "why": "numa_node = -1"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"numa_node": node, "bound": False, "why": "no allowed CPU on the node"}
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "bound": True, "cpus": len(cpus)}
    except Exception as e:  # no sysfs / no nvidia-smi: run unbound
        return {"numa_node": None, "bound": False, "why": f"{type(e).__name__}: {e}"[:120]}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md clocks line)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm (oracle port)
def _cpu_machine(args):
    """
    Reference control flow for one machine: Model.predict in batches of 32 (models.py:289-300) + diff.py:350-444 arithmetic.
    Returns the seconds of the ARITHMETIC only (imports, weight initialisation and data generation are outside the timer).
    """
    m, rows = args
    from oracle import anomaly_math as am
    from oracle import keras_math as km

    spec = km.ff_hourglass_spec(T)
    w = km.init_ff_weights(spec, np.random.default_rng(2000 + m))
    X = np.random.default_rng(1000 + m).random((rows, T))
    y = X.copy()
    sc, mn = am.minmax_fit(y)
    feat = np.full(T, 0.1)
    t0 = time.perf_counter()
    pred = km.ff_predict(spec, w, X, batch_size=32)
    am.anomaly_arrays(pred, y, sc, mn, feat, 0.05)
    return time.perf_counter() - t0


def cpu_one_core(rows: int, machines: int = 2):
    """The scalar port on ONE core, warm: windows/s over the summed arithmetic time of `machines` machines."""
    _cpu_machine((0, 256))  # imports + first-call overheads
    secs = [_cpu_machine((m, rows)) for m in range(machines)]
    return machines * rows / sum(secs), sum(secs)


_POOL = None


def _worker_init():
    try:  # one BLAS thread per worker process, whatever the library read from the environment
        import threadpoolctl

        threadpoolctl.threadpool_limits(1)
    except Exception:
        pass


def cpu_pool(workers: int):
    """
    Persistent worker pool (created and warmed outside any timed region).  Workers are SPAWNED with single-threaded BLAS: forked
    children of a parent that already initialised a 128-thread OpenBLAS each bring up their own 128 threads, and the arm then
    measures oversubscription (round 1: 1.7 M vs 8.0 M windows/s on two boxes with the same core count).
    """
    global _POOL
    if _POOL is None and workers > 1:
        for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[var] = "1"
        import multiprocessing
        from concurrent.futures import ProcessPoolExecutor

        _POOL = ProcessPoolExecutor(max_workers=workers, mp_context=multiprocessing.get_context("spawn"), initializer=_worker_init)
        list(_POOL.map(_cpu_machine, [(m, 64) for m in range(4 * workers)]))  # import numpy/pandas in every worker
    return _POOL


def cpu_windows_per_sec(n_machines: int, rows: int, workers: int):
    """Oracle port on `workers` host processes (one machine at a time each, like the reference's one-pod-per-machine)."""
    jobs = [(m, rows) for m in range(n_machines)]
    pool = cpu_pool(workers)
    t0 = time.perf_counter()
    if pool is None:
        for j in jobs:
            _cpu_machine(j)
    else:
        list(pool.map(_cpu_machine, jobs))
    dt = time.perf_counter() - t0
    return n_machines * rows / dt, dt


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    host = host_info()
    cores = host["usable_cores"]  # worker processes: never more than the cgroup quota allows to run at once
    per_step_machines = 2 * cores
    cpu_pool(cores)
    times = []
    for _ in range(args.warmup):
        cpu_windows_per_sec(per_step_machines, args.rows, cores)
    for _ in range(args.steps):
        v, dt = cpu_windows_per_sec(per_step_machines, args.rows, cores)
        times.append(dt)
    total = args.steps * per_step_machines * args.rows
    value = total / sum(times)
    sample = f"{per_step_machines} machines x {args.rows} rows per step ({cores} worker processes, 1 BLAS thread each) of the {args.machines}-machine workload"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "windows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.machines, args.rows, args.gpus),
        "note": ("reference-restated CPU oracle (NumPy batch-32 predict loop + diff.py arithmetic), not TensorFlow and not the reference's diff.py: "
                 "neither is installable / present on the GPU box; each step is a bounded sample of the configured workload"),
        "cpu_baseline": {"value": value, "unit": "windows/s", "cores": cores, "kind": "port", "sample": sample, "host": host},
        "e2e": {"value": value, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    if _POOL is not None:
        _POOL.shutdown()


def workload_config(machines, rows, world, variant=None):
    """The `config` object: identical for both arms (the reference arm runs bounded samples of the same workload)."""
    cfg = {"workload": "configs[1]: 1000 machines x 64-tag feedforward_hourglass AE, batched predict+anomaly score",
           "machines_per_gpu": machines, "rows_per_machine": rows, "tags": T, "parallelism": f"machines sharded over {world} GPU(s), no data-path collective",
           "l2": "inputs+outputs per step = 15.5 GB >> 126 MB L2 (no flush needed)"}
    if variant is not None:
        cfg["kernel_variant"] = variant
    return cfg


# ------------------------------------------------------------------------------------------------ GPU arm
def dump_outputs(out, total_rows, dest):
    """
    Writes what a caller of the hot path receives (every output array of one step) as <dest>/<name>.npy, float32, on the same
    seeded sample of rows for every array and every run, so that the outputs of two builds can be compared array by array.
    """
    import torch

    os.makedirs(dest, exist_ok=True)
    per_row = sum(t[0].numel() * t.element_size() for t in out.values())
    rows = np.sort(np.random.default_rng(0).choice(total_rows, size=min(total_rows, DUMP_BYTES // per_row), replace=False))
    idx = torch.from_numpy(rows).to(next(iter(out.values())).device)
    for name, t in out.items():
        np.save(os.path.join(dest, f"{name}.npy"), t.index_select(0, idx).cpu().numpy())


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout: libraries (NCCL prints its version banner there) get stderr instead."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--machines", type=int, default=1000, help="machines per GPU")
    ap.add_argument("--rows", type=int, default=10000, help="rows per machine")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", type=int, default=0, help="0 auto, 1 fp32 CUDA cores, 2 tcgen05")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-machines", type=int, default=150, help="machines in the one-core cpu_baseline sample (~10 s of CPU work)")
    ap.add_argument("--secondary", type=int, default=1, help="0: skip the configs[2]/[3]/[4] block")
    ap.add_argument("--numa", type=int, default=1, help="0: do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write rank 0's outputs of the last timed step (a fixed sample of rows) to DIR/<name>.npy")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs --impl ours: the reference arm keeps no outputs")
        run_reference_arm(args, rank, world)
        return

    numa = bind_to_gpu_numa_node(local_rank) if args.numa else {"bound": False, "why": "--numa 0"}
    import torch

    import __graft_entry__ as ge
    from gordo_components_b200 import engine, fleet

    if rank == 0:
        ge.build()
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    from gordo_components_b200.machine.model.factories.feedforward_autoencoder import feedforward_hourglass

    spec = feedforward_hourglass(T)  # the package's own factory: 64-53-43-32-32-43-53-64, tanh hidden, linear out
    M, R = args.machines, args.rows
    # machine assignment: rank 0 decides, NCCL broadcasts (weak scaling: every rank gets M machines of its own)
    assign = fleet.assign_machines(M * world, world, rank, dist)
    assert len(assign) == M

    eng = engine.FFEngine(spec.dims, spec.acts, spec.l1)
    dev = eng.device
    g = torch.Generator(device=dev).manual_seed(1000 + int(assign[0]))
    x = torch.rand((M * R, T), generator=g, device=dev)
    y = x + 0.02 * torch.randn((M * R, T), generator=g, device=dev)
    params = fleet.random_glorot_params(eng, M, g)
    jobs_h = engine.uniform_jobs(M, R)
    jobs = engine.jobs_to_device(jobs_h, dev)
    scale, _ = eng.minmax_fit(jobs, M, R, y, M)
    feat = torch.rand((M, T), generator=g, device=dev) * 0.2 + 0.05
    agg = torch.rand((M,), generator=g, device=dev) * 0.1 + 0.01
    out = {}
    step = lambda: eng.infer_score(params, jobs, M, R, x, y, scale, feat, agg, out=out, variant=args.variant)  # noqa: E731

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    torch.cuda.synchronize()
    ev[0].record()
    for i in range(args.steps):
        step()
        ev[i + 1].record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    elapsed_ms = ev[0].elapsed_time(ev[-1])
    per_launch_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    if rank == 0 and args.dump_outputs:
        dump_outputs(out, M * R, args.dump_outputs)
    t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms_max = float(t.item())
    windows_per_step = M * R * world
    value = windows_per_step * args.steps / (elapsed_ms_max * 1e-3)

    # ---- strong scaling: the SAME M machines split over the ranks (BASELINE: "1k machines at 1/2/4/8 B200") ----------
    Ms = len(fleet.partition(M, world)[rank])
    jobs_s = engine.jobs_to_device(engine.uniform_jobs(Ms, R), dev)
    step_s = lambda: eng.infer_score(params, jobs_s, Ms, R, x, y, scale, feat, agg, out=out, variant=args.variant)  # noqa: E731
    for _ in range(3):
        step_s()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    es0.record()
    for _ in range(args.steps):
        step_s()
    es1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ts = torch.tensor([es0.elapsed_time(es1)], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
    strong_ms = float(ts.item()) / args.steps
    step()  # the weak-scaling outputs again (the summary below reads them)

    # ---- e2e: host buffers through the fleet API, copies inside the timed region ------------------------------
    e2e = fleet.time_e2e(eng, params, jobs_h, x, y, scale, feat, agg, steps=args.e2e_steps, variant=args.variant)
    te = torch.tensor([e2e["ms_per_step"]], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = windows_per_step / (float(te.item()) * 1e-3)

    # ---- after the timed region: gather one summary per machine over NCCL (checksum of the scores) -----------
    summary = out["total-anomaly-confidence"].view(M, R).amax(dim=1)
    gathered = fleet.gather_summaries(summary, world, dist)

    # ---- the other BASELINE configurations: EVERY rank runs its share at the same time (at N = 8 these are configs[2] and
    # configs[3] at spec: 1 000 / 256 machines over 8 GPUs), device time = max over ranks, host-side request rates summed
    peaks, peak_kind = measured_peaks()
    secondary = None
    if args.secondary:
        from benchmarks import secondary as sec

        del out, x, y  # 15 GB of headline buffers are no longer needed
        torch.cuda.empty_cache()
        secondary = {}
        for key, fn in (("configs[3]", lambda: sec.lstm_share(torch, engine, peaks=peaks)), ("configs[2]", lambda: sec.fit_share(torch, engine, fleet)),
                        ("configs[4]", lambda: sec.server_shape(torch, engine, fleet))):
            if dist is not None:
                dist.barrier()
            side_clocks = ClockSampler(local_rank) if key == "configs[3]" else None  # the LSTM share is power bound: its clock belongs to its number
            if side_clocks is not None:
                side_clocks.start()
            try:
                res = fn()
            except Exception as e:  # a failing side measurement must not take the headline line with it
                res = {"error": f"{type(e).__name__}: {e}"[:300]}
            if side_clocks is not None:
                res["clocks"] = side_clocks.stop()
            if dist is not None and "error" not in res:
                if "ms" in res:  # device-timed shares: whole job = all ranks' units over the slowest rank's time
                    tm = torch.tensor([res["ms"]], device=dev, dtype=torch.float64)
                    dist.all_reduce(tm, op=dist.ReduceOp.MAX)
                    scale = res["ms"] / float(tm.item()) * world
                    res["ms"] = float(tm.item())
                    for k in ("windows_per_s", "row_epochs_per_s", "algorithmic_tflops"):
                        if k in res:
                            res[k] *= scale
                    res["aggregate"] = f"{world} ranks x this share, time = max over ranks"
                    if "frac_of_bf16_sustained_peak" in res:  # per GPU
                        res["frac_of_bf16_sustained_peak"] *= scale / world
                        res["tensor_pipe_frac"] *= scale / world
                else:  # request rates measured on the host: sum of the ranks' rates, rank 0's latencies
                    tv = torch.tensor([res["requests_per_s"], res["windows_per_s"], res["all_in_flight"]["windows_per_s"]], device=dev, dtype=torch.float64)
                    dist.all_reduce(tv, op=dist.ReduceOp.SUM)
                    res["requests_per_s"], res["windows_per_s"], res["all_in_flight"]["windows_per_s"] = (float(v) for v in tv)
                    res["aggregate"] = f"sum over {world} ranks (each serves its own resident fleet); latencies are rank 0's"
            secondary[key] = res

    if rank == 0:
        achieved = M * R * BYTES_PER_WINDOW / (float(np.mean(per_launch_ms)) * 1e-3) / 1e9
        # scalar port: one process, one machine at a time, warm; per the contract only at N=1 (other ranks would disturb the host cores)
        cpu_v1, cpu_dt1 = cpu_one_core(R, args.cpu_machines) if world == 1 else (None, 0.0)
        vname = eng_variant_name(args.variant, eng)
        line = {
            "metric": METRIC, "value": value, "unit": "windows/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": elapsed_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if vname == "fma" else "tf32x3", "data": "synthetic",
            "config": workload_config(M, R, world, vname),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                         # dram__bytes_read+write per window from the committed ncu --set full capture of this kernel, times the windows of one launch
                         "traffic": int(M * R * NCU_DRAM_BYTES_PER_WINDOW[vname]),
                         "traffic_source": NCU_SOURCE[vname] + ", scaled per window to this launch", "peak_source": f"MEASURED_PEAKS.json ({peak_kind})", "algorithmic_bytes_per_window": BYTES_PER_WINDOW,
                         "kernel_ms_mean": float(np.mean(per_launch_ms)), "kernel_ms_min": float(np.min(per_launch_ms))},
            "cpu_baseline": {"value": cpu_v1, "unit": "windows/s", "cores": 1, "kind": "port", "host": host_info(),
                             "sample": (f"{args.cpu_machines} machines x {R} rows, NumPy oracle (batch-32 predict loop + diff.py arithmetic), warm, arithmetic only: {cpu_dt1:.1f} s"
                                        if world == 1 else "timed at N=1 only (see the N=1 line)")},
            "e2e": {"value": e2e_value, "unit": "windows/s", "h2d_bytes_per_step": e2e["h2d_bytes"], "d2h_bytes_per_step": e2e["d2h_bytes"],
                    "ms_per_step": float(te.item()), "api": "gordo_components_b200.fleet.anomaly_many (pinned host buffers)",
                    "rank0_h2d_gbs": e2e["h2d_bytes"] / (e2e["ms_per_step"] * 1e6), "rank0_d2h_gbs": e2e["d2h_bytes"] / (e2e["ms_per_step"] * 1e6), "numa": numa},
            "strong": {"value": M * R / (strong_ms * 1e-3), "unit": "windows/s", "ms_per_step": strong_ms, "machines_total": M, "machines_per_gpu": Ms,
                       "note": "the same fleet split over the ranks (strong scaling); `value` above is weak scaling (M machines per GPU)"},
            "secondary": secondary,
            "gpu_launches": args.steps,
            "clocks": clocks,
            "score_checksum": float(gathered.double().sum().item()) if gathered is not None else None,
        }
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def eng_variant_name(variant, eng):
    variant &= 0xFF
    if variant == 1:
        return "fma"
    if variant == 2:
        return "tcgen05"
    from gordo_components_b200 import _cabi
    import ctypes as C

    return "tcgen05" if _cabi.load_library().gb_ffae_tc_supported(C.byref(eng.net)) == 0 else "fma"


if __name__ == "__main__":
    main()
