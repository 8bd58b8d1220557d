#!/usr/bin/env python
"""Benchmark of the exact-inference hot path (see the contract in the task brief).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload grid10x10|asia_1m|dag50]
                    [--rows R] [--impl b200|reference] [--no-extras] [--no-cpu-baseline]
                    [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of synthetic evidence rows:
`rows` independent exact-inference queries (same query variables, same evidence
variables, different observed states) per GPU.  Multi-GPU = one process per GPU
(torchrun), evidence rows sharded across ranks (weak scaling: `rows` per GPU), the only
collective is the final gather of the posteriors on rank 0 (NCCL), inside the timed step
(`sorobn_b200.sharding.ShardedProgram`, the product's torchrun path).

Rank 0 prints ONE JSON line:
  value      rows/s over all GPUs with evidence codes already resident in HBM
  e2e        the same metric with HOST (pinned) buffers: H2D of the evidence codes, every
             kernel, (N > 1: the NCCL gather,) D2H of the posteriors, per step
  roofline   algorithmic HBM bytes of the step kernels / their device time vs measured peak
  cpu_baseline  N = 1 only: the reference's own pandas operators (oracle/_ref, kind "reference")
             on a bounded sample of the same rows, with the numpy oracle port beside it
  extra      the other BASELINE.json configs, bounded to a few seconds each:
             alarm_single_query (configs[0]), asia_1m (configs[1]), dag50 (configs[3]; strong
             scaling: 1M rows split over the N GPUs), gibbs (configs[4]; 10k chains x 10k
             iterations per GPU)

`--impl reference` times the CPU arm instead: the reference's `pointwise_mul` / `sum_out`
(oracle/_ref, copied from /root/reference by oracle/build_ref.py) driven in min-fill order, one
process per host core, a bounded sample of the same workload per step.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "exact-inference queries/sec"
UNIT = "queries/s"
ALARM_QUERY = ("Burglary", {"John calls": True, "Mary calls": True})  # BASELINE.json configs[0]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="grid10x10")
    ap.add_argument("--rows", type=int, default=0, help="evidence rows per GPU per step (0 = workload default)")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows per core of the CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the `extra` block (the other BASELINE configs)")
    ap.add_argument("--dump", default="", help="write per-launch timings (JSON) here")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the posteriors of the last timed step to DIR/posterior.npy (float32 [Q, rows], rank "
                         "order; beyond 64 MB a fixed, seeded sample of the rows, kept in row order)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the posteriors of the b200 arm")
    return args


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """Write each array [Q, rows] as DIR/<name>.npy (float32).  When they exceed DUMP_BYTES in all,
    the same fixed, seeded sample of rows (columns) is taken from every array."""
    arrays = {k: np.asarray(v, dtype=np.float32) for k, v in arrays.items()}
    n = next(iter(arrays.values())).shape[1]
    row_bytes = sum(a.shape[0] * 4 for a in arrays.values())
    if row_bytes * n > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // row_bytes, replace=False))
        arrays = {k: a[:, keep] for k, a in arrays.items()}
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, f"{k}.npy"), np.ascontiguousarray(a))


# ------------------------------------------------------------------ clocks sampling
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU through NVML every ~2 ms.  The thread
    is started early (NVML init takes longer than the timed region); `begin()` / `end()`
    bracket the timed region and only samples taken in between are reported."""

    def __init__(self, index: int):
        self.index = index
        self.sm, self.reasons_seen = [], 0
        self.max_sm = None
        self._stop = threading.Event()
        self._ready = threading.Event()
        self._active = False
        self._ok = False
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        self._ready.wait(timeout=20)

    def _run(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self._ok = True
            self._ready.set()
            while not self._stop.is_set():
                if self._active:
                    self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    try:
                        self.reasons_seen |= int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                    except Exception:
                        self.reasons_seen |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self._stop.wait(0.002)
        except Exception:
            self._ok = False
            self._ready.set()

    def begin(self):
        self.sm, self.reasons_seen = [], 0
        self._active = True

    def end(self):
        self._active = False

    def close(self):
        self._stop.set()
        self._thread.join(timeout=6)

    def summary(self):
        if not self._ok or not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": [], "samples": 0}
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                "hw_power_brake_slowdown": 0x80}
        reasons = [n for n, b in bits.items() if self.reasons_seen & b]
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.max_sm, "reasons": reasons,
                "samples": len(self.sm)}


# ------------------------------------------------------------------------ CPU legs
# Two CPU implementations of the same path, both driven in the device program's min-fill order
# (the planner is imported only to obtain that order; it helps the CPU arm -- the reference's own
# set-iteration order is OOM-killed on the grid):
#   "reference"  oracle/_ref: the reference's own pandas operators (bayes_net.py:54-256)
#   "port"       oracle/ve_oracle.py: the dense numpy restatement
_CPU_STATE = {}


def ref_available() -> bool:
    from oracle import build_ref

    return build_ref.available()


def _cpu_state(workload, kind):
    key = (workload, kind)
    if key not in _CPU_STATE:
        from sorobn_b200 import planner, workloads

        wl = workloads.WORKLOADS[workload]()
        bn = wl.build()
        net = bn._compiled
        plan = planner.build_plan(net, [net.index[q] for q in wl.query], [net.index[e] for e in wl.evidence])
        order = [net.names[v] for v in plan.order]
        if kind == "reference":
            from oracle import build_ref, ref_driver

            ref = build_ref.import_reference()
            impl = (ref, ref_driver.build_workload(ref, wl), ref_driver)
        else:
            from oracle import ve_oracle

            impl = (ve_oracle, ve_oracle.dense_from_pandas(bn.P, bn.parents, bn.nodes), None)
        _CPU_STATE[key] = (wl, net, order, impl)
    return _CPU_STATE[key]


def _cpu_worker(args):
    """Answer rows [lo, hi); network / plan setup is cached per process (the warm-up map pays
    for it), so the timed map measures inference only."""
    workload, kind, codes, lo, hi = args
    wl, net, order, impl = _cpu_state(workload, kind)
    acc = 0.0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # pandas PerformanceWarning inside the reference
        for b in range(lo, hi):
            ev = {v: net.domains[net.index[v]][codes[i, b]] for i, v in enumerate(wl.evidence)}
            if kind == "reference":
                ref, ref_bn, drv = impl
                acc += float(drv.ordered_query(ref, ref_bn, wl.query, ev, order).iloc[0])
            else:
                ve, dn, _ = impl
                acc += float(ve.query(dn, *wl.query, event=ev, order=order)[1].reshape(-1)[0])
    return acc


def _cpu_warm(args):
    _cpu_state(*args)
    time.sleep(0.2)
    return os.getpid()


class CpuArm:
    """A pool of single-threaded worker processes, one per usable host core."""

    def __init__(self, workload, kind, n_procs):
        import multiprocessing as mp

        self.workload, self.kind, self.n_procs = workload, kind, max(1, n_procs)
        for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
            os.environ[var] = "1"  # numpy's own thread pools would oversubscribe the cores
        self.pool = mp.get_context("spawn").Pool(self.n_procs)
        # warm every worker (imports, network build, plan): chunksize 1 and as many tasks as
        # workers, each sleeping briefly so that no worker takes two
        self.pool.map(_cpu_warm, [(workload, kind)] * self.n_procs, chunksize=1)

    def rate(self, codes, n_rows):
        """rows/s over `n_rows` rows spread evenly over the workers."""
        n_rows = min(n_rows, codes.shape[1])
        bounds = np.linspace(0, n_rows, self.n_procs + 1).astype(int)
        jobs = [(self.workload, self.kind, codes, int(bounds[i]), int(bounds[i + 1]))
                for i in range(self.n_procs) if bounds[i + 1] > bounds[i]]
        t0 = time.perf_counter()
        self.pool.map(_cpu_worker, jobs, chunksize=1)
        return n_rows / (time.perf_counter() - t0)

    def close(self):
        self.pool.close()
        self.pool.join()


def effective_cores() -> int:
    """Host cores this process may actually use: the smallest of the CPU count, the scheduler
    affinity mask and the cgroup CPU quota (containers often expose 128 CPUs with a quota of 8)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as f:
                parts = f.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    n = min(n, max(1, int(int(parts[0]) / int(parts[1]))))
            else:
                quota = int(parts[0])
                if quota > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
                        n = min(n, max(1, quota // int(g.read().split()[0])))
            break
        except Exception:
            continue
    return max(1, n)


# rows per core of one CPU sample (sized for ~1 s per step with the reference, ~1 s with the port)
CPU_ROWS_PER_CORE = {
    "reference": {"grid10x10": 2, "asia_1m": 40, "dag50": 2},
    "port": {"grid10x10": 512, "asia_1m": 8192, "dag50": 256},
}


def cpu_baseline_block(workload, codes, cores, rows_per_core=0):
    """The CPU numbers printed beside the GPU line: the reference (when oracle/_ref travelled) and
    the numpy port, each on `cores` processes over a bounded sample of the same rows."""
    out = {}
    for kind in (["reference"] if ref_available() else []) + ["port"]:
        rpc = rows_per_core or CPU_ROWS_PER_CORE[kind].get(workload, 2)
        n = min(codes.shape[1], rpc * cores)
        arm = CpuArm(workload, kind, cores)
        try:
            arm.rate(codes, max(cores, n // 4))  # warm-up pass
            rate = arm.rate(codes, n)
        finally:
            arm.close()
        out[kind] = {"value": rate, "rows": n}
    kind = "reference" if "reference" in out else "port"
    what = {"reference": "oracle/_ref: the reference's own pandas pointwise_mul / sum_out (bayes_net.py:54-256) "
                         "driven in the device program's min-fill order",
            "port": "oracle/ve_oracle.py: numpy port of the reference's variable elimination, same min-fill order"}
    block = {"value": out[kind]["value"], "unit": UNIT, "cores": cores, "kind": kind,
             "sample": f"first {out[kind]['rows']} evidence rows of the same batch, {cores} processes ({what[kind]})"}
    if kind == "reference":
        block["port"] = {"value": out["port"]["value"], "unit": UNIT, "cores": cores,
                         "sample": f"first {out['port']['rows']} rows, {cores} processes ({what['port']})"}
    return block


def alarm_reference_latency(reps=30):
    """configs[0]: wall time of the reference's own `query` (bayes_net.py:796-875) for the Alarm query."""
    if not ref_available():
        return None
    from oracle import build_ref
    from sorobn_b200 import examples

    ref = build_ref.import_reference()
    bn = examples.build(examples.NETWORKS["alarm"], cls=ref.BayesNet)
    q, ev = ALARM_QUERY
    ts = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for _ in range(reps + 3):
            t = time.perf_counter()
            ans = bn.query(q, event=ev)
            ts.append(time.perf_counter() - t)
    return {"ms": 1e3 * float(np.median(ts[3:])), "reps": reps, "answer": {str(k): float(v) for k, v in ans.items()},
            "impl": "oracle/_ref BayesNet.query(algorithm='exact'), one host core"}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            with open(path) as f:
                return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(workload: str):
    """Per-launch DRAM traffic of the dominant kernel from the committed ncu capture."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        try:
            with open(path) as f:
                return json.load(f).get(workload)
        except Exception:
            return None
    return None


def workload_config(wl, rows, world):
    """The `config` both arms print (identical dicts: same workload, same rows per step per GPU)."""
    return {"workload": wl.name, "description": wl.description, "rows_per_gpu": rows, "global_rows": rows * world,
            "query": list(wl.query), "n_evidence": len(wl.evidence), "elimination_order": "min-fill"}


# ------------------------------------------------------------------ reference arm
def run_reference(args, rank, world):
    if rank != 0:
        return
    from sorobn_b200 import workloads

    wl = workloads.WORKLOADS[args.workload]()
    bn = wl.build()
    cores = effective_cores()
    kind = "reference" if ref_available() else "port"
    rpc = args.cpu_rows or CPU_ROWS_PER_CORE[kind].get(args.workload, 2)
    sample = rpc * cores
    rows = args.rows or wl.default_rows
    codes = wl.codes(bn, max(sample, 512 * cores), seed=1000)  # the rows rank 0 of the GPU arm answers
    arm = CpuArm(args.workload, kind, cores)
    try:
        for _ in range(max(0, args.warmup)):
            arm.rate(codes, sample)
        rates = [arm.rate(codes, sample) for _ in range(max(1, args.steps))]
    finally:
        arm.close()
    value = float(np.mean(rates))
    what = ("oracle/_ref = the reference's own pandas pointwise_mul / sum_out (bayes_net.py:54-256, copied unmodified "
            "from /root/reference by oracle/build_ref.py) driven in min-fill order; the reference's own set-order "
            "elimination is OOM-killed on the grid" if kind == "reference" else
            "oracle/ve_oracle.py, numpy port of the reference's variable elimination (oracle/_ref did not travel)")
    cpu = {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": f"{sample} evidence rows ({rpc} per core) of the same workload per step, {cores} single-threaded "
                     f"processes; {what}"}
    if kind == "reference":
        port = CpuArm(args.workload, "port", cores)
        try:
            n_port = CPU_ROWS_PER_CORE["port"].get(args.workload, 256) * cores
            port.rate(codes, n_port // 4)
            cpu["port"] = {"value": port.rate(codes, n_port), "unit": UNIT, "cores": cores,
                           "sample": f"{n_port} rows, {cores} processes (oracle/ve_oracle.py numpy port)"}
        finally:
            port.close()
    extra = {}
    if not args.no_extras:
        lat = alarm_reference_latency()
        if lat:
            extra["alarm_single_query"] = lat
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sample / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(wl, rows, world),
        "sample_rows_per_step": sample,
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "extra": extra,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------- B200 arm
class Timer:
    """Device timing of `steps` calls of fn(): CUDA events on the current stream, a barrier +
    synchronize on both sides, optional L2 flush (a 256 MB write) before every timed call."""

    def __init__(self, torch, dist, distributed, dev):
        self.torch, self.dist, self.distributed, self.dev = torch, dist, distributed, dev
        self._flush = None

    def barrier(self):
        if self.distributed:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def flush_buffer(self):
        if self._flush is None:
            self._flush = self.torch.empty(256 * 1024 * 1024, dtype=self.torch.uint8, device=self.dev)
        return self._flush

    def device_ms(self, fn, steps, flush):
        torch = self.torch
        if not flush:
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.barrier()
            start.record()
            for _ in range(steps):
                fn()
            end.record()
            self.barrier()
            return start.elapsed_time(end)
        total = 0.0
        for _ in range(steps):
            self.flush_buffer().fill_(1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.barrier()
            s.record()
            fn()
            e.record()
            self.barrier()
            total += s.elapsed_time(e)
        return total

    def wall_s(self, fn, steps):
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        self.barrier()
        return time.perf_counter() - t0

    def max_over_ranks(self, *vals):
        t = self.torch.tensor(list(vals), dtype=self.torch.float64, device=self.dev)
        if self.distributed:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]


def exact_workload(ctx, wl, rows, steps, warmup, want_profile=False, counts=None, keep_output=False):
    """Time one exact-inference workload on this rank's GPU (+ gather when distributed).
    Returns a dict on rank 0 (None elsewhere): device-timed and end-to-end numbers, and with
    `keep_output` the posteriors [Q, global rows] of the last device-timed step."""
    import torch

    from sorobn_b200 import engine, planner, sharding

    tm, rank, world, local_rank, dev = ctx["timer"], ctx["rank"], ctx["world"], ctx["local_rank"], ctx["dev"]
    bn = wl.build(device=local_rank)
    net = bn._compiled
    plan = planner.build_plan(net, [net.index[q] for q in wl.query], [net.index[e] for e in wl.evidence])
    prog = engine.Program(plan, device=local_rank)
    prog.reserve(rows)
    reserved = prog.info()["reserved_rows"]
    assert reserved >= rows, f"scratch for {rows} rows does not fit (got {reserved})"
    n_ev, Q = prog.n_ev, prog.Q
    codes_host = engine.PinnedArray((max(n_ev, 1), rows), np.uint8)
    codes_host.array[:n_ev] = wl.codes(bn, rows, seed=1000 + rank)
    out_host = engine.PinnedArray((Q, rows), np.float32)
    distributed = world > 1
    step_bytes = plan.bytes_per_row() * rows
    flush = step_bytes < 512e6  # working set could sit in the 126 MB L2: flush between steps

    if distributed:
        sp = sharding.ShardedProgram(prog, Q, n_ev, rows, dst=0, device=dev)
        sp.upload(codes_host.array[:n_ev])
        d_out = sp.d_out
        device_step = lambda: sp.run_resident(rows)  # noqa: E731
        host_step = lambda: sp.run_host(codes_host.array[:n_ev], rows, counts=counts, blocks=True)  # noqa: E731
        e2e_api = ("sharding.ShardedProgram.run_host(blocks=True): pinned H2D, sbn_program_run_device, NCCL gather, "
                   "D2H on rank 0 into per-rank [Q, rows] blocks")
    else:
        d_ev = torch.from_numpy(codes_host.array).to(dev)
        d_out = torch.empty((Q, rows), dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream().cuda_stream
        device_step = lambda: prog.run_device(d_ev.data_ptr(), rows, rows, d_out.data_ptr(), rows, stream)  # noqa: E731
        host_step = lambda: prog.run(codes_host.array[:n_ev], rows, out=out_host.array)  # noqa: E731
        e2e_api = "sbn_program_run_host (pinned host buffers)"

    for _ in range(warmup):
        device_step()
    tm.barrier()
    launches0 = prog.info()["launches"]
    dev_ms = tm.device_ms(device_step, steps, flush)
    launches = prog.info()["launches"] - launches0
    posterior = None
    if keep_output and rank == 0:  # copied before the end-to-end steps below run the rows again
        posterior = (sp.gathered.transpose(0, 1).reshape(Q, -1) if distributed else d_out).clone()
    for _ in range(max(1, warmup // 2)):
        host_step()
    e2e_s = tm.wall_s(host_step, steps)
    dev_ms, e2e_s = tm.max_over_ranks(dev_ms, e2e_s)

    sums = d_out[:, :rows].sum(dim=0)
    ok = bool(torch.isfinite(sums).all() and ((sums - 1).abs() < 1e-4).all())
    if rank != 0:
        return None
    same = True
    if not distributed:
        same = bool(np.array_equal(out_host.array, d_out.cpu().numpy()))
    ms_per_step = dev_ms / steps
    total_rows = rows * world if counts is None else int(sum(counts))
    res = {
        "plan": plan, "prog": prog, "bn": bn, "codes_host": codes_host, "rows": rows, "flush": flush, "posterior": posterior,
        "ms_per_step": ms_per_step, "value": total_rows / (ms_per_step * 1e-3),
        "e2e_ms_per_step": 1e3 * e2e_s / steps, "e2e_value": total_rows / (e2e_s / steps),
        "h2d": int(n_ev * rows) * world, "d2h": int(Q * rows * 4) * world, "e2e_api": e2e_api,
        "launches": int(launches) * world, "ok": ok, "same": same, "total_rows": total_rows,
        # bytes the launches as issued move: paired steps keep their intermediate in registers
        "bytes_issued_per_row": plan.bytes_per_row() - prog.info()["pair_bytes_saved_per_row"],
    }
    res["whole_step_frac"] = (res["bytes_issued_per_row"] * rows / (ms_per_step * 1e-3) / 1e9) / measured_peak()[0]
    if want_profile and not distributed:
        d_ev_ptr = d_ev.data_ptr()
        prof = None
        for _ in range(3):
            t = prog.profile(d_ev_ptr, rows, rows, d_out.data_ptr(), rows, stream)
            prof = t if prof is None else np.minimum(prof, t)
        res["profile_ms"] = prof
    return res


def summarise_exact(res, wl):
    """JSON block of one `extra` exact workload."""
    plan = res["plan"]
    return {
        "workload": wl.name, "rows_per_gpu": res["rows"], "global_rows": res["total_rows"],
        "value": res["value"], "unit": UNIT, "ms_per_step": res["ms_per_step"],
        "e2e": {"value": res["e2e_value"], "unit": UNIT, "ms_per_step": res["e2e_ms_per_step"],
                "h2d_bytes_per_step": res["h2d"], "d2h_bytes_per_step": res["d2h"], "api": res["e2e_api"]},
        "algorithmic_bytes_per_row": plan.bytes_per_row(), "bytes_per_row_as_issued": res["bytes_issued_per_row"],
        "hbm_roofline_frac_whole_step": res["whole_step_frac"],
        "launches_per_step": res["launches"] // max(1, res.get("steps", 1)),
        "l2": "flushed (256 MB write) between timed steps" if res["flush"] else "not flushed (step streams >> 126 MB)",
        "checks": {"posteriors_sum_to_one": res["ok"], "host_path_equals_device_path": res["same"]},
    }


def gibbs_extra(ctx, steps, warmup):
    """configs[4]: Gibbs sampling on the 100-node grid, 10k chains x 10k iterations per GPU (the
    chain frequencies are gathered on rank 0 with NCCL when N > 1)."""
    import torch
    import torch.distributed as dist

    from sorobn_b200 import engine, workloads

    tm, rank, world, local_rank, dev = ctx["timer"], ctx["rank"], ctx["world"], ctx["local_rank"], ctx["dev"]
    wl = workloads.grid10x10()
    bn = wl.build(device=local_rank)
    net = bn._compiled
    n_chains, n_iter = 10_000, 10_000
    q_ids = [net.index[q] for q in wl.query]
    ev_ids = [net.index[e] for e in wl.evidence]
    cycle = [net.index[v] for v in sorted(set(bn.nodes) - set(wl.evidence))]
    sampler = engine.GibbsSampler(net, q_ids, ev_ids, cycle, device=local_rank)
    codes = wl.codes(bn, 1, seed=77)
    codes = np.ascontiguousarray(np.repeat(codes, n_chains, axis=1))  # every chain: the same event
    gathered = torch.empty((world, sampler.Q, n_chains), dtype=torch.float32, device=dev) if rank == 0 else None

    def step():
        freq = sampler.run(codes, n_chains, n_iter, seed=1234 + rank)
        if world > 1:
            t = torch.from_numpy(freq).to(dev)
            dist.gather(t, list(gathered.unbind(0)) if rank == 0 else None, dst=0)
        return freq

    for _ in range(max(1, warmup // 2)):
        freq = step()
    s = tm.wall_s(step, steps)
    (s,) = tm.max_over_ranks(s)
    if rank != 0:
        return None
    # sanity: the mean over chains approaches the exact posterior of that event
    exact = bn.query_many(*wl.query, events=wl.events(1, seed=77, bn=bn)).to_numpy()[0]
    est = freq.mean(axis=1)
    updates = n_chains * n_iter * world
    return {"chains_per_gpu": n_chains, "iterations": n_iter, "n_cycle": len(cycle), "ms_per_run": 1e3 * s / steps,
            "value": updates / (s / steps), "unit": "variable updates/s (whole job, host in/out included)",
            "max_abs_error_of_chain_mean_vs_exact": float(np.max(np.abs(est - exact))),
            "api": "sbn_sampler_run_host (one chain per evidence row)" + ("; NCCL gather of frequencies" if world > 1 else "")}


def alarm_extra(local_rank):
    """configs[0] on the GPU side: `BayesNet.query` for the Alarm query, cold (first call: planning,
    program creation, table launches, run) and warm (median of 200 calls)."""
    from sorobn_b200 import examples

    q, ev = ALARM_QUERY
    bn = examples.build(examples.NETWORKS["alarm"], device=local_rank)
    t = time.perf_counter()
    ans = bn.query(q, event=ev)
    cold = time.perf_counter() - t
    ts = []
    for _ in range(200):
        t = time.perf_counter()
        bn.query(q, event=ev)
        ts.append(time.perf_counter() - t)
    return {"cold_ms": 1e3 * cold, "warm_ms": 1e3 * float(np.median(ts)), "reps": 200,
            "answer": {str(k): float(v) for k, v in ans.items()},
            "impl": "sorobn_b200.BayesNet.query (float64 single-event program, sbn_program_run_host_f64)"}


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    from sorobn_b200 import planner, sharding, workloads

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed and not dist.is_initialized():
        # stdout carries the one JSON line: NCCL prints its version banner to fd 1 when the
        # communicator is created, so fd 1 points at stderr until that has happened
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    ctx = {"timer": Timer(torch, dist, distributed, dev), "rank": rank, "world": world, "local_rank": local_rank,
           "dev": dev}
    wl = workloads.WORKLOADS[args.workload]()
    rows = args.rows or wl.default_rows

    clocks = ClockSampler(local_rank)
    clocks.begin()
    res = exact_workload(ctx, wl, rows, args.steps, args.warmup, want_profile=True, keep_output=bool(args.dump_outputs))
    clocks.end()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"posterior": res["posterior"].cpu().numpy()})
    clock_summary = clocks.summary()
    clocks.close()

    # ---- the other BASELINE configs, a few seconds each (every rank takes part in the collectives)
    extra = {}
    if not args.no_extras:
        k, w = max(3, min(args.steps, 5)), 3
        for name in ("asia_1m", "dag50"):
            if name == wl.name:
                continue
            wl2 = workloads.WORKLOADS[name]()
            counts = None
            rows2 = wl2.default_rows
            if name == "dag50" and world > 1:  # configs[3]: 1M queries sharded over the GPUs (strong scaling)
                counts = [s.stop - s.start for s in (sharding.row_shard(wl2.default_rows, r, world) for r in range(world))]
                rows2 = counts[rank]
            r2 = exact_workload(ctx, wl2, rows2, k, w, counts=counts)
            if rank == 0:
                r2["steps"] = k
                extra[name] = summarise_exact(r2, wl2)
                extra[name]["scaling"] = ("strong (1M rows over all GPUs)" if counts else
                                          "weak (rows per GPU fixed)" if world > 1 else "single GPU")
        g = gibbs_extra(ctx, 3, 2)
        if rank == 0:
            extra["gibbs"] = g
            extra["alarm_single_query"] = {"b200": alarm_extra(local_rank)}

    if rank == 0:
        plan, prog = res["plan"], res["prog"]
        net = res["bn"]._compiled
        ms_per_step = res["ms_per_step"]
        peak, peak_src = measured_peak()
        roofline = {"bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src,
                    "whole_step_frac": res["whole_step_frac"]}
        if "profile_ms" in res:
            # per-launch CUDA events (same stream, outside the graph: a few us of overhead each), used
            # only for the SHARE of the step the step kernels take; the time itself is the timed region's
            prof = res["profile_ms"]
            sb = plan.step_bytes_per_row()
            kern = float(sum(ms for ms, st in zip(prof[:-1], plan.steps) if st.kind == planner.KIND_BATCHED))
            share = kern / float(prof.sum()) if prof.sum() > 0 else 1.0
            kernel_ms = ms_per_step * share
            # paired steps (csrc/sbn_pair.h) keep their intermediate in registers: those bytes are not moved
            # and do not count -- the figure is what the launches as issued have to read and write
            info = prog.info()
            kernel_bytes = float(sum(sb) - info["pair_bytes_saved_per_row"]) * rows
            achieved = kernel_bytes / (kernel_ms * 1e-3) / 1e9
            traffic = ncu_traffic(wl.name) if rows == wl.default_rows else None
            n_batched = int(sum(1 for st in plan.steps if st.kind == planner.KIND_BATCHED))
            # per kernel family: bytes its launches move / their share of the timed step (roles from the engine)
            roles = prog.step_roles()
            fam_of = {1: "sbn_step_tiled", 2: "sbn_pair_kernel", 3: "sbn_pair_kernel", 4: "sbn_triple_kernel", 5: "sbn_triple_kernel"}
            fams = {}
            mid = 0  # bytes per row of the intermediate a fused launch keeps on chip
            for i, st in enumerate(plan.steps):
                role = int(roles[i])
                fam = fam_of.get(role)
                if fam is None:
                    continue
                d = fams.setdefault(fam, {"launches": 0, "bytes_per_row": 0, "ms": 0.0})
                d["ms"] += float(prof[i])
                if role in (2, 4):    # first step of a fused launch: its output is never written ...
                    mid = 4 * int(np.prod(st.cards, dtype=np.int64))
                    d["bytes_per_row"] += sb[i] - mid
                elif role in (3, 5):  # ... nor read back by the second
                    d["bytes_per_row"] += sb[i] - mid
                else:
                    d["bytes_per_row"] += sb[i]
                d["launches"] += 1 if role in (1, 2, 4) else 0
            for d in fams.values():
                d["ms"] *= ms_per_step / float(prof.sum())
                d["achieved_gbs"] = d["bytes_per_row"] * rows / (d["ms"] * 1e-3) / 1e9 if d["ms"] > 0 else None
                d["frac"] = d["achieved_gbs"] / peak if d["ms"] > 0 else None
                d["share_of_step"] = d["ms"] / ms_per_step
            # headline = the dominant kernel family, per launch; the aggregate over every step kernel beside it
            dom_name, dom = max(fams.items(), key=lambda kv: kv[1]["ms"])
            dom_traffic = None
            if traffic and traffic.get("by_kernel", {}).get(dom_name):
                tk = traffic["by_kernel"][dom_name]
                dom_traffic = tk["dram_bytes"] / max(1, tk["launches"])
            roofline.update({
                "kernel": f"{dom_name} ({dom['launches']} launches per step, {dom['share_of_step']:.0%} of the step)",
                "achieved": dom["achieved_gbs"], "frac": dom["frac"],
                "algorithmic_bytes_per_launch": dom["bytes_per_row"] * rows / max(1, dom["launches"]),
                "avg_launch_ms": dom["ms"] / max(1, dom["launches"]),
                "traffic": dom_traffic,
                "all_step_kernels": {
                    "achieved": achieved, "frac": achieved / peak, "algorithmic_bytes_per_step": kernel_bytes,
                    "kernel_ms_per_step": kernel_ms, "kernel_share_of_step": share,
                    "launches_per_step": n_batched - info["pairs"], "fused_launches": info["pairs"],
                    "bytes_per_row_one_launch_per_step": int(sum(sb)),
                    "bytes_per_row_as_issued": int(sum(sb) - info["pair_bytes_saved_per_row"]),
                    "traffic": (traffic or {}).get("dram_bytes_per_step"),
                },
                "by_kernel": fams, "traffic_detail": traffic,
            })
            if args.dump:
                with open(args.dump, "w") as f:
                    json.dump({"workload": wl.name, "rows": rows, "step_ms": [float(x) for x in prof],
                               "step_bytes_per_row": sb,
                               "steps": [{"kind": st.kind, "cx": st.cx, "cards": list(st.cards),
                                          "inputs": [("B" if fct.batched else "t") + str(int(np.prod([net.card[v] for v in fct.vars])) if fct.vars else 1)
                                                     + (f"e{len(fct.ev)}" if fct.ev else "") for fct, _, _ in st.inputs]}
                                         for st in plan.steps]}, f)
        else:
            achieved = res["bytes_issued_per_row"] * rows / (ms_per_step * 1e-3) / 1e9
            roofline.update({"kernel": "whole step (per-launch profile only at N = 1)", "achieved": achieved,
                             "frac": achieved / peak, "traffic": None})

        cpu = None
        if not args.no_cpu_baseline and not distributed:
            cores = effective_cores()
            cpu = cpu_baseline_block(wl.name, np.ascontiguousarray(res["codes_host"].array[:prog.n_ev, :min(rows, 512 * cores)]),
                                     cores, args.cpu_rows)
            if not args.no_extras:
                lat = alarm_reference_latency()
                if lat:
                    extra.setdefault("alarm_single_query", {})["reference_cpu"] = lat

        cfg = workload_config(wl, rows, world)
        line = {
            "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "plan": {
                "parallelism": f"rows sharded x{world}; NCCL gather of posteriors",
                "elimination_steps": len(plan.steps), "max_factor_entries_per_row": plan.max_factor_per_row(),
                "algorithmic_bytes_per_row": plan.bytes_per_row(), "bytes_per_row_as_issued": res["bytes_issued_per_row"],
                "l2": ("flushed (256 MB write) between timed steps" if res["flush"] else
                       f"not flushed: each step streams {plan.bytes_per_row() * rows / 1e9:.2f} GB of factors >> 126 MB L2"),
            },
            "e2e": {"value": res["e2e_value"], "unit": UNIT, "h2d_bytes_per_step": res["h2d"],
                    "d2h_bytes_per_step": res["d2h"], "ms_per_step": res["e2e_ms_per_step"], "api": res["e2e_api"]},
            "gpu_launches": res["launches"],
            "roofline": roofline,
            "cpu_baseline": cpu,
            "clocks": clock_summary,
            "checks": {"posteriors_sum_to_one": res["ok"], "host_path_equals_device_path": res["same"]},
            "extra": extra,
        }
        print(json.dumps(line), flush=True)

    if distributed:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
