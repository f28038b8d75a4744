#!/usr/bin/env python
"""bench.py — headline benchmark of the registrators/ hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One *alignment* is BASELINE.json configs[1]: a synthetic 64-beam 120 000-point scan against a
500 000-point submap (106 784 target points with normals after the caller-side CalculateNormals),
point-to-plane IcpFast with the iteration count fixed at 30 (convergence test disabled on both
arms, SURVEY.md section 8d), i.e. SetInputTarget + SetInputSource + Align including the k-d tree
rebuild.  One *step* is a BATCH of --batch (64) such alignments per GPU — BASELINE.json
configs[3]'s per-GPU share (512 pairs on 8 GPUs) — pushed through the batched entry point
sm_align_pairs by --host-threads (2) host threads over --pipelines (16) matcher instances.

* `value`  : alignments/s, clouds already resident in HBM (device pointers), K timed steps (one window
             unless --windows splits them; then the median per-step time), device time (CUDA events), max
             over ranks, pose all-gather included.
* `e2e`    : the same through host buffers (pinned host memory -> H2D inside the timed region,
             result records read back, all-gather included), another K timed steps.
* --dump-outputs DIR : the rcs, poses and scores that the last timed step of each path returned
             (`icp_*`, `icp_e2e_*`, `ndt_*`, `ndt_gicp_*`) as float64 .npy files; the inputs are seeded, so
             they are the same from run to run.
* roofline : dominant kernel (transform + k-NN), algorithmic bytes of SURVEY.md section 8d over the
             CUDA-event time of its launches, measured here with one alignment in flight; the
             16-in-flight regime of `value` is reported beside it (kernels of different alignments
             overlap, so the serial sum of one alignment's launches exceeds ms_per_step / batch).
* cpu_baseline / --impl reference : the CPU oracle (a restatement of the reference's libnabo +
             Eigen path; the reference itself cannot be compiled in this image) on the host cores
             this process may use (sched_getaffinity / cgroup quota), one thread per physical core,
             and again with 6 threads (the reference's hard-coded NDT thread count, ndt.cc:32).
* extra    : BASELINE.json configs[2] (Ndt) and configs[4] (NdtWithGicp loop-closure pairs, sharded
             over the ranks, pose all-gather) measured the same way, CPU oracle beside them at N=1.

One process per GPU (torchrun for N > 1); every rank aligns its own pairs (weak scaling, no
data-path collective) and the resulting poses are all-gathered over NCCL.
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
# more hardware work queues than the default 8, so that the per-pipeline streams do not alias
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

N_SOURCE = 120_000
N_SUBMAP = 500_000
ITERATIONS = 30
BYTES_PER_POINT_ITER = 64           # SURVEY.md 8d: whole iteration
BYTES_KNN_PER_POINT = 40            # of which the k-NN kernel: 16 src + 16 matched + 8 write
# dram__bytes_read + dram__bytes_write of ONE launch of icp_knn_kernel from the committed
# `ncu --set full` capture (profiles/r02_ncu_full_icp_knn_final.txt; ncu flushes the caches
# before the launch, so this is the cold figure; the steady state of an alignment is lower)
NCU_TRAFFIC_BYTES = 6_438_400
KNN_KERNEL = "icp_knn_kernel"
METRIC = "scan-pair alignments/sec (120k->500k pts, 30 ICP iters)"
UNIT = "alignments/s"
NDT_GICP_PAIRS = 2048               # BASELINE.json configs[4]


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def make_workload(pair: int):
    """(source (Ns,3) f64, submap (500k,3) f64, perturbation) for pair index `pair`."""
    cache = f"/tmp/sm_b200_bench_pair{pair}.npz"
    if os.path.exists(cache):
        try:
            z = np.load(cache)
            return z["src"], z["sub"], z["P"]
        except Exception:  # noqa: BLE001  (a concurrently written cache file)
            pass
    from staticmapping_b200 import synth
    t0 = time.time()
    scene = synth.make_scene(0)
    sub = synth.submap(scene, seed=pair, n_points=N_SUBMAP).astype(np.float64)
    scan = synth.lidar_scan(scene, (2.0, 0.0, 0.0), seed=10_000 + pair).astype(np.float64)
    P = synth.perturbation(pair)
    src = synth.apply_se3(np.linalg.inv(P), scan + np.array([2.0, 0.0, 0.0]))
    src = src.astype(np.float32).astype(np.float64)   # clouds enter as float (InnerPointType)
    assert src.shape == (N_SOURCE, 3) and sub.shape == (N_SUBMAP, 3)
    try:
        tmp = f"{cache}.{os.getpid()}.tmp.npz"
        np.savez(tmp, src=src, sub=sub, P=P)
        os.replace(tmp, cache)
    except OSError:
        pass
    log(f"[bench] workload pair {pair} generated in {time.time() - t0:.1f}s")
    return src, sub, P


# ------------------------------------------------------------------------------ host resources
def usable_cpus():
    """(logical CPUs this process may run on, physical cores among them, cgroup quota or None)."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
    except AttributeError:
        cpus = list(range(os.cpu_count() or 1))
    cores = set()
    for c in cpus:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                cores.add(f.read().strip())
        except OSError:
            cores.add(str(c))
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, per = f.read().split()
            if q != "max":
                quota = float(q) / float(per)
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except (OSError, ValueError):
            pass
    return len(cpus), len(cores), quota


def cpu_threads():
    """One OpenMP thread per usable physical core (one per SMT sibling was measured 3.6x slower),
    capped by the cgroup CPU quota."""
    logical, phys, quota = usable_cpus()
    n = phys
    if quota is not None:
        n = max(1, min(n, int(quota)))
    return max(1, n), {"logical_cpus": logical, "physical_cores": phys, "cgroup_quota": quota}


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def oracle_module(threads):
    """The CPU arms: thread count and placement are fixed BEFORE libgomp starts (torchrun exports
    OMP_NUM_THREADS=1, which would silently make this a single-thread baseline)."""
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib
    oracle_lib.set_num_threads(threads)
    return oracle_lib


def cpu_time_alignments(O, src, tp, tn, min_reps, max_seconds):
    """Full oracle alignments (fixed 30 iterations) until `min_reps` are done and, beyond that,
    while less than `max_seconds` have been spent.  Returns (seconds per alignment, the last alignment's result)."""
    ts = []
    while len(ts) < min_reps or (sum(ts) < max_seconds and len(ts) < 4 * min_reps):
        t0 = time.perf_counter()
        r = O.icp_fast_align(src, tp, tn, max_iteration=ITERATIONS, disable_convergence_check=True)
        ts.append(time.perf_counter() - t0)
        assert r["rc"] == 1 and r["iterations"] == ITERATIONS
    return ts, r


def window_steps(steps, windows):
    """The `steps` timed steps split into at most `windows` windows whose sizes differ by at most one."""
    w = min(windows, steps)
    return [steps // w + (k < steps % w) for k in range(w)]


def dump_outputs(path, arrays):
    """--dump-outputs: one float64 .npy per returned array."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def workload_config(n_target, batch):
    return {"workload": "configs[1] alignments (single 120k-pt scan -> 500k-pt submap, point-to-plane ICP, "
                        "30 iters) in batches of configs[3]'s per-GPU share",
            "n_source": N_SOURCE, "n_submap_raw": N_SUBMAP, "n_target_after_prep": int(n_target),
            "iterations": ITERATIONS, "knn_epsilon": 3.16, "dist_outlier_ratio": 0.7,
            "convergence_check": "disabled", "alignments_per_step": batch}


def run_reference(args, rank, world):
    """--impl reference: the CPU path of the reference (oracle restatement, kind "port"; `oracle/_ref`
    does not exist because the reference cannot be compiled here) on the host cores of the box.
    Rank 0 alone runs it, on all the cores it may use; the figure does not depend on --gpus."""
    if rank != 0:
        return
    threads, res = cpu_threads()
    O = oracle_module(threads)
    src, sub, _ = make_workload(0)
    tp, tn = O.calculate_normals(sub)
    cpu_time_alignments(O, src, tp, tn, max(1, min(args.warmup, 2)), 0.0)
    ts, r = cpu_time_alignments(O, src, tp, tn, args.steps, 0.0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"icp_ok": [r["rc"]], "icp_poses": r["result"][None], "icp_scores": [r["score"]]})
    total = float(np.sum(ts))
    value = len(ts) / total
    cores = O.num_threads()
    cfg = workload_config(tp.shape[0], args.batch)
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(ts), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "cpu_model": cpu_model(), "host": res,
                         "sample": f"{len(ts)} steps of ONE alignment each (a bounded sample of the "
                                   f"{args.batch}-alignment batch the GPU arm runs per step; 120k->{tp.shape[0]} pts, "
                                   f"30 fixed iterations, k-d tree rebuilt each time), OpenMP over queries with "
                                   f"{cores} threads (one per usable physical core), rest serial as in the reference",
                         "scope": "whole host CPU of the box, rank 0 only: independent of --gpus"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def stop(self, t_from=None, t_to=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, ln in self.lines:
            if t_from is not None and not (t_from <= ts <= t_to + 0.3):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(smax)) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------ GPU arm
class PairData:
    """One scan pair: device-resident and pinned-host copies of the three clouds."""

    def __init__(self, smb, torch, dev, local_rank, pair):
        self.src, sub, self.P = make_workload(pair)
        tgt = smb.CalculateNormals(sub, device=local_rank)      # target prep on the GPU
        self.tp, self.tn = np.ascontiguousarray(tgt.points), np.ascontiguousarray(tgt.normals)
        self.nt = self.tp.shape[0]
        self.d = [torch.from_numpy(a).to(dev) for a in (self.src, self.tp, self.tn)]
        self.h = [torch.from_numpy(a).pin_memory() for a in (self.src, self.tp, self.tn)]

    def pair(self, host):
        a = self.h if host else self.d
        return {"source": int(a[0].data_ptr()), "target": int(a[1].data_ptr()), "normals": int(a[2].data_ptr()),
                "n_source": N_SOURCE, "n_target": self.nt, "on_device": not host}

    @property
    def h2d_bytes(self):
        return int(self.src.nbytes + self.tp.nbytes + self.tn.nbytes + 128)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64,
                    help="alignments per step and GPU (configs[3]: 512 pairs over 8 GPUs)")
    ap.add_argument("--pipelines", "--inflight", type=int, default=16, dest="pipelines",
                    help="matcher instances (= alignments in flight) per GPU")
    ap.add_argument("--host-threads", type=int, default=2, help="host threads that drive the pipelines")
    ap.add_argument("--windows", type=int, default=1,
                    help="timed windows the --steps steps are split into; the median per-step time is reported "
                         "(each window adds ~2 ms of ramp-up and drain on a B200 at 1000 W, so shorter windows "
                         "lower the figure)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the Ndt / NdtWithGicp records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of each timed path returned as DIR/<name>.npy (float64; "
                         "rank 0's pairs), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.windows < 1:
        ap.error("--steps and --windows must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    import staticmapping_b200 as smb
    from staticmapping_b200 import parallel

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (staticmapping_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    sampler = ClockSampler(local_rank) if local_rank == 0 else None
    if sampler:
        sampler.start()                      # before warm-up: spawning it must not land in a timed window

    # ---- inputs: every pipeline of every rank owns a distinct scan pair ------------------------
    P = max(1, args.pipelines)
    T = max(1, min(args.host_threads, P))
    B = max(1, args.batch)
    data = [PairData(smb, torch, dev, local_rank, rank * P + w) for w in range(P)]
    matchers = []
    for _ in range(P):
        m = smb.IcpFast(local_rank)
        opts = {"max_iteration": ITERATIONS, "disable_convergence_check": 1,
                "knn_queries_per_cta": os.environ.get("SM_B200_KNN_QPC", "1024")}   # many alignments in flight
        m.InitWithXml(opts)
        matchers.append(m)
    streams = [torch.cuda.Stream(device=dev) for _ in range(P)]
    for m, s in zip(matchers, streams):
        m.SetStream(s.cuda_stream)
    tstream = torch.cuda.Stream(device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    gather_ms = []

    def gather_poses(results, scores):
        """the one collective of the path: all-gather of the poses (17 doubles per pair)"""
        if world == 1:
            return None
        rec = parallel.pack_poses(list(results), list(scores))
        t = torch.from_numpy(rec).to(dev)
        out = [torch.empty_like(t) for _ in range(world)]
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); dist.all_gather(out, t); e1.record(); e1.synchronize()
        gather_ms.append(e0.elapsed_time(e1))
        return out

    def run_steps(steps, host):
        """`steps` batches of B alignments through sm_align_pairs: host thread j drives the pipelines
        j, j+T, ... with the pairs j, j+T, ... of the batch.  Device time of the whole region: an
        event before (every pipeline stream waits on it) and one after (it waits on every pipeline),
        plus the all-gather of the last batch's poses.  Returns (ms, what the last step returned for the
        batch: rcs, poses, scores in batch order)."""
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        errors, last = [], [None] * T
        gate = threading.Barrier(T + 1)
        pairs = [data[k % P].pair(host) for k in range(B)]

        def body(j):
            ms = matchers[j::T]
            mine = pairs[j::T]
            try:
                gate.wait()
                for _ in range(steps):
                    last[j] = smb.AlignPairs(ms, mine)
            except Exception as e:  # noqa: BLE001
                errors.append(e)

        threads = [threading.Thread(target=body, args=(j,)) for j in range(T)]
        for t in threads:
            t.start()
        torch.cuda.synchronize()
        e0.record(tstream)
        for s in streams:
            s.wait_event(e0)
        gate.wait()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        for s in streams:
            ev = torch.cuda.Event(); ev.record(s); tstream.wait_event(ev)
        e1.record(tstream)
        e1.synchronize()
        rcs, res, sc = np.empty(B), np.empty((B, 4, 4)), np.empty(B)
        for j, (rcs_j, res_j, sc_j) in enumerate(last):
            rcs[j::T], res[j::T], sc[j::T] = rcs_j, res_j, sc_j
        gather_poses(res, sc)                 # once per window, inside the reported time
        return e0.elapsed_time(e1) + (gather_ms[-1] if world > 1 else 0.0), (rcs, res, sc)

    # ---- warm-up (graphs captured, allocations done, all-gather warmed) -------------------------
    run_steps(args.warmup, False)
    run_steps(args.warmup, True)
    w0 = matchers[0]
    w0.SetInputTargetDevice(data[0].d[1].data_ptr(), data[0].d[2].data_ptr(), data[0].nt)
    w0.SetInputSourceDevice(data[0].d[0].data_ptr(), N_SOURCE)
    _, res_check = w0.Align(np.eye(4))
    per_align_launches = w0.GetAlignInfo()["kernel_launches"] + 3
    barrier()
    gather_ms.clear()
    t_mark0 = sampler.mark() if sampler else None
    windows = window_steps(args.steps, args.windows)
    # ---- timed: device-resident inputs -------------------------------------------------------
    win_dev = []
    for n in windows:
        barrier()
        ms, dev_out = run_steps(n, False)
        barrier()
        win_dev.append(max_over_ranks(ms))
    # ---- timed: host buffers through the public API (H2D inside) ---------------------------
    win_e2e = []
    for n in windows:
        barrier()
        ms, e2e_out = run_steps(n, True)
        barrier()
        win_e2e.append(max_over_ranks(ms))
    t_mark1 = sampler.mark() if sampler else None
    outputs = {}
    for prefix, (rcs, res, sc) in (("icp", dev_out), ("icp_e2e", e2e_out)):
        outputs.update({f"{prefix}_ok": rcs, f"{prefix}_poses": res, f"{prefix}_scores": sc})
    ms_dev_step = float(np.median([ms / n for ms, n in zip(win_dev, windows)]))
    ms_e2e_step = float(np.median([ms / n for ms, n in zip(win_e2e, windows)]))
    gpu_launches = per_align_launches * B * args.steps
    allgather_incl_wait_ms = float(np.median(gather_ms)) if gather_ms else 0.0
    allgather_ms = 0.0
    if world > 1:                     # the collective alone (ranks aligned by a barrier first): 17 doubles per pair
        rec = torch.zeros((B, parallel.POSE_RECORD), dtype=torch.float64, device=dev)
        outl = [torch.empty_like(rec) for _ in range(world)]
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); dist.all_gather(outl, rec); e1.record(); e1.synchronize()
        allgather_ms = e0.elapsed_time(e1)

    # ---- latency: one alignment in flight, L2 flushed before each -----------------------------
    for m in matchers:
        m.InitWithXml({"knn_queries_per_cta": 0})        # one alignment in flight: one query per thread

    def timed_serial(step_fn, k, stream):
        total_ms = 0.0
        with torch.cuda.stream(stream):
            for _ in range(k):
                flush.zero_()
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                step_fn()
                e1.record(stream)
                e1.synchronize()
                total_ms += e0.elapsed_time(e1)
        return total_ms

    d0 = data[0]

    def step_device():
        w0.SetInputTargetDevice(d0.d[1].data_ptr(), d0.d[2].data_ptr(), d0.nt)
        w0.SetInputSourceDevice(d0.d[0].data_ptr(), N_SOURCE)
        return w0.Align(np.eye(4))

    def step_host():
        w0._check(w0._lib.sm_set_input_target(w0._h, d0.h[1].data_ptr(), d0.h[2].data_ptr(), d0.nt), "SetInputTarget")
        w0._check(w0._lib.sm_set_input_source(w0._h, d0.h[0].data_ptr(), N_SOURCE), "SetInputSource")
        return w0.Align(np.eye(4))

    timed_serial(step_device, 2, streams[0])
    lat_steps = 10
    ms_lat_dev = timed_serial(step_device, lat_steps, streams[0]) / lat_steps
    ms_lat_host = timed_serial(step_host, lat_steps, streams[0]) / lat_steps
    # ---- dominant-kernel timing: extra profiled alignments, events around every launch -----------
    w0.InitWithXml({"profile_kernels": 1})
    timed_serial(step_device, 1, streams[0])
    prof = {"knn": 0.0, "accum": 0.0, "finish": 0.0, "prologue": 0.0, "n": 0}
    for _ in range(3):
        timed_serial(step_device, 1, streams[0])
        info = w0.GetAlignInfo()
        prof["knn"] += info["ms_knn"]; prof["accum"] += info["ms_accum"]
        prof["finish"] += info["ms_finish"]; prof["prologue"] += info["ms_prologue"]
        prof["n"] += 1
    w0.InitWithXml({"profile_kernels": 0})
    clocks = sampler.stop(t_mark0, t_mark1) if sampler else None

    value = B * world / (ms_dev_step * 1e-3)
    e2e_value = B * world / (ms_e2e_step * 1e-3)
    knn_ms = prof["knn"] / prof["n"] / ITERATIONS          # average launch duration
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = BYTES_KNN_PER_POINT * N_SOURCE / (knn_ms * 1e-3) / 1e9
    iter_ms = (prof["knn"] + prof["accum"] + prof["finish"]) / prof["n"]
    per_gpu_rate = value / world
    roofline = {"bound": "hbm", "kernel": KNN_KERNEL, "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": NCU_TRAFFIC_BYTES,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
                "avg_launch_ms": knn_ms, "bytes_per_launch": BYTES_KNN_PER_POINT * N_SOURCE,
                "regime": "ONE alignment in flight: CUDA events around every launch of 3 extra profiled "
                          "alignments run right after the timed windows, same stream and inputs. The working set "
                          "is L2-resident and the kernel is a divergent, latency-bound tree walk; with "
                          f"{P} alignments in flight (the regime of `value`) kernels of different alignments overlap "
                          "and the per-alignment serial sum below exceeds ms_per_step / alignments_per_step",
                "per_alignment_ms": {k: prof[k] / prof["n"] for k in ("prologue", "knn", "accum", "finish")},
                "iteration_bytes_frac": (BYTES_PER_POINT_ITER * N_SOURCE * ITERATIONS / (iter_ms * 1e-3) / 1e9) / peak,
                # the same algorithmic bytes at the measured many-in-flight rate of one GPU
                "in_flight_regime": {"alignments_in_flight": P,
                                     "knn_bytes_frac": (BYTES_KNN_PER_POINT * N_SOURCE * ITERATIONS * per_gpu_rate / 1e9) / peak,
                                     "iteration_bytes_frac": (BYTES_PER_POINT_ITER * N_SOURCE * ITERATIONS * per_gpu_rate / 1e9) / peak},
                # informational (SURVEY 8d second figure, NOT the graded fraction): bytes the traversal
                # itself touches per query — 14 nodes x 9 B + an 8-point bucket x 24 B + the 64 B above
                "traversal_inclusive_frac": (382 * N_SOURCE / (knn_ms * 1e-3) / 1e9) / peak}

    cfg = workload_config(d0.nt, B)
    cfg.update({"pipelines_per_gpu": P, "host_threads": T, "windows": len(windows), "steps_per_window": windows,
                "entry_point": "sm_align_pairs (one call per host thread and step)",
                "l2": f"{P} distinct pairs in flight per GPU (combined working set ~{25 * P} MB vs 126 MB L2), every "
                      "alignment re-uploads / re-reads its clouds and rebuilds its tree; the latency figures flush "
                      "L2 (256 MiB memset) before every alignment",
                "timed_window_ms": {"device_resident": win_dev, "host_buffers": win_e2e}})
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_dev_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": cfg,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": d0.h2d_bytes * B,
                "d2h_bytes_per_step": (128 + 400) * B, "ms_per_step": ms_e2e_step},
        "latency": {"ms_per_alignment_device": ms_lat_dev, "ms_per_alignment_host_buffers": ms_lat_host,
                    "in_flight": 1, "icp_iterations_per_s": ITERATIONS / (iter_ms * 1e-3)},
        "gpu_launches": gpu_launches, "clocks": clocks, "roofline": roofline,
        "allgather_ms": allgather_ms,
        "allgather_incl_rank_skew_ms": allgather_incl_wait_ms,   # as it happened inside the timed windows (waits for the slowest rank)
    }
    if world > 1:
        # clocks were sampled on local rank 0 only (one nvidia-smi, started before warm-up)
        out["clocks_scope"] = "GPU of local rank 0"

    # ---- extra: configs[2] (Ndt) and configs[4] (NdtWithGicp, sharded, pose all-gather) ----------
    if not args.no_extra:
        try:
            out["extra"] = run_extra(args, smb, torch, dist, parallel, dev, rank, local_rank, world, P, outputs)
        except Exception as e:  # noqa: BLE001
            # the headline measurement above is complete: with one rank a failure of the side records must not
            # lose it (with several ranks the others are inside collectives, so the error has to propagate)
            if world > 1:
                raise
            out["extra"] = {"error": f"{type(e).__name__}: {e}"}

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu_legs(out, d0, res_check)
        except Exception as e:  # noqa: BLE001  (same reasoning: keep the GPU line and what was measured so far)
            out.setdefault("cpu_baseline", {})["error"] = f"{type(e).__name__}: {e}"
    if "extra" in out:
        for rec in out["extra"].values():
            if isinstance(rec, dict):
                rec.pop("result_check", None)
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(out), flush=True)
    # orderly teardown: drain the GPU and destroy the engine handles before the interpreter
    # (and torch's CUDA context) goes away
    torch.cuda.synchronize()
    for m in matchers:
        m.SetStream(0)
        m.__del__()
    del matchers, w0
    torch.cuda.synchronize()
    if world > 1:
        dist.destroy_process_group()


def cpu_legs(out, d0, res_check):
    """cpu_baseline (all usable physical cores, and the reference's 6 threads), the parity spot check of the
    benchmarked configuration and the oracle beside the extra records: rank 0 at N = 1 only."""
    threads, res = cpu_threads()
    O = oracle_module(threads)
    ts, _ = cpu_time_alignments(O, d0.src, d0.tp, d0.tn, 3, 10.0)
    # parity spot check of the benchmarked configuration against the oracle
    o = O.icp_fast_align(d0.src, d0.tp, d0.tn, max_iteration=ITERATIONS, disable_convergence_check=True)
    E = np.linalg.inv(o["result"]) @ res_check
    out["parity_vs_oracle"] = {"dt_m": float(np.linalg.norm(E[:3, 3])),
                               "dr_rad": float(np.arccos(np.clip((np.trace(E[:3, :3]) - 1) / 2, -1, 1)))}
    cores = O.num_threads()
    out["cpu_baseline"] = {
        "value": len(ts) / float(np.sum(ts)), "unit": UNIT, "cores": cores, "kind": "port",
        "cpu_model": cpu_model(), "host": res,
        "sample": f"{len(ts)} full alignments of the same workload (30 fixed iterations, tree rebuilt each "
                  f"time), one at a time, OpenMP over queries with {cores} threads (one per usable physical core)"}
    O.set_num_threads(6)                  # the reference's own hard-coded thread count (ndt.cc:32)
    ts6, _ = cpu_time_alignments(O, d0.src, d0.tp, d0.tn, 2, 6.0)
    out["cpu_baseline"]["six_threads"] = {"value": len(ts6) / float(np.sum(ts6)), "unit": UNIT, "cores": 6,
                                          "sample": f"{len(ts6)} alignments"}
    O.set_num_threads(threads)
    if "extra" in out:
        cpu_extra(O, out["extra"])


def run_extra(args, smb, torch, dist, parallel, dev, rank, local_rank, world, pairs_per_rank, outputs):
    """Ndt (configs[2]) and NdtWithGicp (configs[4]: 2048 loop-closure candidate pairs sharded over the
    ranks, poses all-gathered) on the same clouds: float scan + raw 500k submap.  What the last timed batch
    of each returned goes into `outputs`."""
    from staticmapping_b200 import InnerCloud
    npairs = 4
    clouds = []
    for k in range(npairs):
        src, sub, _ = make_workload(rank * pairs_per_rank + k)
        clouds.append((InnerCloud(src.astype(np.float32)), InnerCloud(sub.astype(np.float32))))
    out = {}
    for name, cls, total_pairs in (("ndt", smb.Ndt, 512 * world), ("ndt_gicp", smb.NdtWithGicp, NDT_GICP_PAIRS)):
        ms_ = []
        for k in range(npairs):
            m = cls(local_rank)
            m.SetInputSource(clouds[k][0]); m.SetInputTarget(clouds[k][1])
            ms_.append(m)
        guesses = [np.eye(4)] * npairs
        smb.AlignBatch(ms_, guesses)                                   # warm-up (allocations)
        ok, res1 = ms_[0].Align(np.eye(4))
        info = ms_[0].GetAlignInfo()
        torch.cuda.synchronize()
        t0 = time.perf_counter(); ms_[0].Align(np.eye(4)); lat = time.perf_counter() - t0
        share = max(npairs, total_pairs // world)
        if world > 1:                                                  # warm the collective on this record size
            t = torch.zeros((share, parallel.POSE_RECORD), dtype=torch.float64, device=dev)
            dist.all_gather([torch.empty_like(t) for _ in range(world)], t)
            dist.barrier()
        torch.cuda.synchronize()
        # wall time, barrier to the end of the pose all-gather: these optimisers are driven from the host
        # (Newton / BFGS steps with a read-back each), so device events would miss the host part
        done, t0 = 0, time.perf_counter()
        all_res, all_sc = [], []
        while done < share:
            oks, res = smb.AlignBatch(ms_, guesses)
            all_res.extend(res); all_sc.extend(m.GetFitnessScore() for m in ms_)
            done += npairs
        outputs.update({f"{name}_ok": oks, f"{name}_poses": res, f"{name}_scores": all_sc[-npairs:]})
        ag_ms = 0.0
        if world > 1:
            rec = parallel.pack_poses(all_res, all_sc)                 # every pose of the shard: 136 B per pair
            t = torch.from_numpy(rec).to(dev)
            outl = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(outl, t)
            torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        if world > 1:
            tt = torch.tensor([secs], dtype=torch.float64, device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            secs = float(tt.item())
            dist.barrier()                                             # the collective alone, ranks aligned
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(); dist.all_gather(outl, t); e1.record(); e1.synchronize()
            ag_ms = e0.elapsed_time(e1)
        rec = {"pairs_total": done * world, "pairs_per_s": done * world / secs,
               "ms_per_alignment_one_in_flight": lat * 1e3, "instances_in_flight_per_gpu": npairs,
               "allgather_ms": ag_ms, "iterations": info["iterations"], "evaluations": info["evaluations"],
               "timing": "wall clock from a barrier to the end of the pose all-gather, max over ranks",
               "result_check": res1.tolist()}
        if name == "ndt":
            nbar = info["mean_neighbors"]
            rec.update({"mean_neighbors": nbar, "config": "configs[2]: NDT l=1.0 m, 120k -> 500k pts",
                        "algorithmic_bytes_per_derivative_evaluation": N_SOURCE * (12 + 27 * 8 + nbar * 136)})
        else:
            rec.update({"config": f"configs[4]: {NDT_GICP_PAIRS} loop-closure candidate pairs NDT+GICP sharded over "
                                  f"{world} GPU(s), pose all-gather", "bfgs_evaluations": info["profiled_iterations"]})
        out[name] = rec
        for m in ms_:
            m.__del__()
    return out


def cpu_extra(O, extra):
    """the oracle beside the Ndt / NdtWithGicp records (one alignment each: ~0.4 s / ~1.2 s)"""
    src, sub, _ = make_workload(0)
    s32, t32 = src.astype(np.float32), sub.astype(np.float32)
    for name, fn in (("ndt", O.ndt_align), ("ndt_gicp", O.ndt_gicp_align)):
        if name not in extra:
            continue
        t0 = time.perf_counter(); o = fn(s32, t32); dt = time.perf_counter() - t0
        E = np.linalg.inv(o["result"]) @ np.array(extra[name]["result_check"])
        extra[name]["cpu_oracle"] = {"s_per_alignment": dt, "pairs_per_s": 1.0 / dt, "threads": O.num_threads()}
        extra[name]["parity_vs_oracle"] = {"dt_m": float(np.linalg.norm(E[:3, 3])),
                                           "dr_rad": float(np.arccos(np.clip((np.trace(E[:3, :3]) - 1) / 2, -1, 1)))}


if __name__ == "__main__":
    main()
