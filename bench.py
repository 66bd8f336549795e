#!/usr/bin/env python
"""bench.py -- TPC-H through the B200 execution engine; headline: q1 SF10 (BASELINE.json configs[1]).

One "step" = one full pass of the hot path over the resident synthetic lineitem table:
  stage 1  scan -> FilterExec -> ProjectionExec -> AggregateExec(Partial) -> hash ShuffleWriter
  stage 2  ShuffleReader -> AggregateExec(FinalPartitioned) -> SortExec -> ShuffleWriter(None)
  stage 3  ShuffleReader -> SortPreservingMergeExec -> ShuffleWriter(None)
exactly the stage shapes Ballista's planner emits for q1 (ballista/scheduler/src/planner.rs:655-670).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
N>1 is launched by the driver under torchrun (one rank per GPU, NCCL); every rank owns SF10 worth
of lineitem rows (weak scaling: the global table is SF(10*N)), the partial aggregate states are
exchanged with an NCCL all-to-all, and `value` is global rows / max-over-ranks device time.

`--impl reference` times the CPU restatement of the reference path (oracle/, all host threads) on
a bounded sample of the same workload: the reference itself (Rust) cannot be built offline.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SF10_MSF = 10000
ROWS_SF10 = 59_986_052
BYTES_PER_ROW = 78  # Arrow layout of the 7 referenced columns (SURVEY.md 8(d) config 1)
METRIC = "tpch_q1_rows_per_sec"
try:
    START_AFFINITY = os.sched_getaffinity(0)
except Exception:  # pragma: no cover
    START_AFFINITY = None


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ---- clocks ---------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region.  NVML (nvidia_ml_py) is polled in-process every
    2 ms -- the timed region of this benchmark is tens of milliseconds, shorter than one `nvidia-smi -lms` tick;
    nvidia-smi is only the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []
        self.nvml = None
        self.handle = None
        self.sm, self.reasons = [], set()
        self.max_mhz = None
        self.stop_flag = False
        self.t = None

    def _nvml_sample(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40)):
            if r & bit:
                self.reasons.add(name)

    def _nvml_loop(self):
        while not self.stop_flag:
            try:
                self._nvml_sample()
            except Exception:
                break
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.gpu_index
            if vis:
                ids = [x for x in vis.split(",") if x.strip() != ""]
                if self.gpu_index < len(ids) and ids[self.gpu_index].strip().isdigit():
                    phys = int(ids[self.gpu_index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self._nvml_sample()  # at least one sample at the start of the timed region
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return
        except Exception as e:
            self.nvml = None
            log("NVML clock sampling unavailable (", e, "); falling back to nvidia-smi")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu_index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception as e:  # pragma: no cover
            log("clock sampler unavailable:", e)

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.nvml is not None:
            try:
                self._nvml_sample()  # ... and one at its end
            except Exception:
                pass
            self.stop_flag = True
            if self.t:
                self.t.join(timeout=1)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ---- CPU arm (oracle) -------------------------------------------------------------------------------
def usable_cpus() -> int:
    """CPUs this process may actually use: the cgroup quota when there is one (the B200 boxes expose 128
    hardware threads under a 16-CPU quota; oversubscribing it only adds throttling), else os.cpu_count()."""
    n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(quota) // int(period)))
    except Exception:
        pass
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return n


def host_mem_available() -> int:
    """Bytes this process may still allocate: MemAvailable, capped by what the container's memory cgroup (v2 or v1) leaves."""
    avail = 0
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                avail = int(ln.split()[1]) * 1024
    except Exception:
        pass
    for mx, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                    ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            limit = open(mx).read().strip()
            if limit and limit != "max" and int(limit) < (1 << 60):
                avail = min(avail, max(0, int(limit) - int(open(cur).read().strip()))) if avail else max(0, int(limit) - int(open(cur).read().strip()))
        except Exception:
            pass
    return avail


def cpu_q1(msf: int, row_begin: int, row_end: int, threads: int, steps: int, warmup: int):
    """q1 over lineitem rows [row_begin, row_end) of the SF(msf/1000) table on the CPU oracle: `threads` map tasks in
    parallel (the reference runs one task per partition on its DedicatedExecutor pool, cpu_bound_executor.rs:94-131).
    Returns (seconds per timed pass, result table)."""
    import oracle_ffi
    from concurrent.futures import ThreadPoolExecutor
    from ballista_b200 import tpch
    eng = oracle_ffi.OracleEngine()     # loads the oracle/liboracle.so the build made: no `make` in a tree that may be read-only
    parts = threads
    rows = row_end - row_begin
    step = (rows + parts - 1) // parts
    res = None
    with ThreadPoolExecutor(threads) as pool:
        list(pool.map(lambda p: eng.tpch_generate("lineitem", msf, p, min(row_end, row_begin + p * step), min(row_end, row_begin + (p + 1) * step),
                                                  tpch.Q1_COLUMNS), range(parts)))
        stages = tpch.q1(n_partitions=min(16, parts))
        times = []
        for it in range(warmup + steps):
            job = f"cpu{it}"
            t0 = time.perf_counter()
            s1 = eng.create_query_stage_exec(job, 1, stages[0].json(job))
            list(pool.map(lambda p: s1.execute_query_stage(p), range(parts)))
            s2 = eng.create_query_stage_exec(job, 2, stages[1].json(job))
            list(pool.map(lambda p: s2.execute_query_stage(p), range(min(16, parts))))
            s3 = eng.create_query_stage_exec(job, 3, stages[2].json(job))
            s3.execute_query_stage(0)
            res = eng.partition_export(job, 3, 0)
            dt = time.perf_counter() - t0
            eng.remove_job_data(job)
            if it >= warmup:
                times.append(dt)
            assert res.num_rows == 4
    eng.close()
    return times, res


PORT_NOTE = ("CPU restatement of the reference path (oracle/liboracle.so, one map task per host thread); the Rust reference cannot be "
             "built offline.  Per core it is about 4x slower than the published Ballista anchor (q1 SF100 in 7.5 s on 8 cores = "
             "80 M rows/s including Parquet decode, BASELINE.md)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = usable_cpus()
    if args.workload != "q1":
        emit({"impl": "reference", "unavailable": f"CPU arm implemented for the q1 headline workload only (asked: {args.workload})"})
        return
    rows = ROWS_SF10  # the FULL configs[1] table, like the GPU arm's per-GPU share
    times, res = cpu_q1(SF10_MSF, 0, rows, threads, args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"q1": res})
    total = sum(times)
    value = rows * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "decimal128/i128",
        "data": "synthetic",
        "config": {"workload": "TPC-H q1 SF10 (BASELINE.json configs[1])", "rows_per_step": rows, "note": PORT_NOTE},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port",
                         "sample": f"q1 over all {rows} lineitem rows of SF10 per step, {threads} map tasks on {threads} threads"},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ---- GPU arm ----------------------------------------------------------------------------------------
def tables_equal(a, b, f64_rtol=0.0) -> bool:
    from util import assert_tables_equal
    try:
        assert_tables_equal(a, b, sort=False, f64_rtol=f64_rtol)
        return True
    except AssertionError as ex:
        log("PARITY MISMATCH:", ex)
        return False


def setup_engine(args):
    """One process per GPU: torch.distributed (NCCL) is the launcher-side plumbing (barriers, the max over ranks);
    the data path's exchange is the engine's own communicator (b200_engine_comm_init)."""
    import torch
    import torch.distributed as dist
    import ballista_b200 as bb
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("--gpus N > 1 must be launched under torchrun (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    eng = bb.GpuExecutionEngine(local_rank, 0, rank, world)
    stream = torch.cuda.Stream(device=device)
    eng.set_stream(stream.cuda_stream)
    if world > 1:
        # fused shuffle (b200_stage_execute_exchange): a window of HBM per executor that the peers' partition scatter kernels
        # store into directly; sized for the largest fixed-width shuffle of the workload
        wgb = args.exchange_window_gb
        if wgb < 0:
            wgb = 0.0 if args.workload == "q1" else 16.0
        if wgb > 0 and not args.no_fused_shuffle:
            eng.set_config("b200.exchange.window_bytes", str(int(wgb * (1 << 30))))
        idt = torch.zeros(128, dtype=torch.uint8, device=device)
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(bb.GpuExecutionEngine.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        eng.comm_init(bytes(idt.cpu().numpy().tobytes()))
    return torch, dist, bb, eng, stream, device, rank, world, local_rank


def run_b200(args):
    if args.workload != "q1":
        return run_workload(args)
    torch, dist, bb, eng, stream, device, rank, world, local_rank = setup_engine(args)
    import pyarrow as pa
    from ballista_b200 import tpch
    from ballista_b200.engine import EXCHANGE_GATHER, EXCHANGE_HASH

    # this rank's slice of the global SF(10*world) lineitem table, generated directly in HBM
    msf = SF10_MSF * world
    r0, r1 = rank * ROWS_SF10, (rank + 1) * ROWS_SF10
    eng.tpch_generate("lineitem", msf, 0, r0, r1, tpch.Q1_COLUMNS)
    P = world
    stages = tpch.q1(n_partitions=P)
    partial_schema = stages[1].plan["input"]["input"]["input"]["schema"]
    final_schema = stages[2].plan["input"]["input"]["schema"]

    agg_ns = [0, 0]  # [elapsed ns, launches] of the fused stage-1 kernel inside the timed region
    exch = {"sent": 0, "recv": 0, "calls": 0}
    trace = os.environ.get("B200_BENCH_TRACE")
    tr = {}

    def _mark(name, t0):
        if trace:
            torch.cuda.synchronize(device)
            tr[name] = tr.get(name, 0.0) + (time.perf_counter() - t0) * 1e3
        return time.perf_counter()

    def step(job, timed=False, table="lineitem"):
        t0 = time.perf_counter()
        pj = [s.json(job) for s in stages]
        if table != "lineitem":
            pj = [j.replace('"table":"lineitem"', f'"table":"{table}"') for j in pj]
        s1 = eng.create_query_stage_exec(job, 1, pj[0])
        s1.execute_query_stage(0)
        if timed:
            for m in s1.collect_plan_metrics():
                if m["name"] == "AggregateExec":
                    agg_ns[0] += m["elapsed_compute_ns"]
                    agg_ns[1] += 1
        s1.release()
        t0 = _mark("stage1", t0)
        if world > 1:
            st = eng.exchange_stage(job, 1, P, partial_schema, EXCHANGE_HASH, 0)
            exch["sent"] += st["sent_bytes"]
            exch["recv"] += st["recv_bytes"]
            exch["calls"] += 1
            t0 = _mark("exchange1", t0)
        s2 = eng.create_query_stage_exec(job, 2, pj[1])
        s2.execute_query_stage(rank)
        s2.release()
        t0 = _mark("stage2", t0)
        out = None
        if world > 1:
            # final merge on rank 0: every rank's stage-2 output (one partition each) goes to the merge task
            st = eng.exchange_stage(job, 2, world, final_schema, EXCHANGE_GATHER, 0)
            exch["sent"] += st["sent_bytes"]
            exch["recv"] += st["recv_bytes"]
            exch["calls"] += 1
            t0 = _mark("gather", t0)
        if rank == 0:
            s3 = eng.create_query_stage_exec(job, 3, pj[2])
            s3.execute_query_stage(0)
            s3.release()
            out = eng.partition_export(job, 3, 0)
        eng.remove_job_data(job)
        _mark("stage3", t0)
        return out

    # ---- warm-up (also settles the aggregate strategy hint) ----
    res = None
    for w in range(max(args.warmup, 3)):
        res = step(f"warm#{w}")
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)

    tr.clear()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.kernel_launches()
    for k in exch:
        exch[k] = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(args.steps):
        res = step(f"step#{k}", timed=True)
    e1.record(stream)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1)
    launches = eng.kernel_launches() - launches0
    exch_timed = dict(exch)   # the e2e passes below go through the same step()
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        lt = torch.tensor([launches], dtype=torch.int64, device=device)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt.item())

    total_rows = ROWS_SF10 * world
    value = total_rows * args.steps / (ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"q1": res})

    if trace:
        print(f"[trace rank {rank}] per-step ms: " + ", ".join(f"{k}={v / args.steps:.3f}" for k, v in tr.items()), file=sys.stderr)

    # ---- end to end: host (pinned) Arrow buffers -> C-ABI -> result on host, every step, at every N ----
    e2e = measure_e2e(eng, bb, pa, torch, dist, step, rank, world, device, steps=max(3, min(args.steps, 5)))

    # ---- parity of the TIMED path's result with the CPU oracle on the same (global) table: untimed ----
    parity = {"checked": False}
    if rank == 0 and not args.no_parity:
        try:
            os.sched_setaffinity(0, START_AFFINITY)
        except Exception:
            pass
        threads = usable_cpus()
        need = total_rows * 100
        if host_mem_available() > need * 1.3:
            t0 = time.perf_counter()
            _, want = cpu_q1(msf, 0, total_rows, threads, steps=1, warmup=0)
            ok = tables_equal(pa.Table.from_batches([res]), pa.Table.from_batches([want]))
            parity = {"checked": True, "equal": ok, "oracle_seconds": time.perf_counter() - t0,
                      "what": f"q1 result of the timed path (N={world}, global SF{10 * world}) == CPU oracle on the same {total_rows} rows, bit-exact"}
        else:
            parity = {"checked": False, "why": f"host memory: need {need >> 30} GiB for the oracle's copy of the global table"}

    line = None
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        kern_s = (agg_ns[0] / max(agg_ns[1], 1)) / 1e9
        alg_bytes = ROWS_SF10 * BYTES_PER_ROW + 4 * (2 * 5 + 13 * 16)
        achieved = alg_bytes / kern_s / 1e9 if kern_s > 0 else 0.0
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "q1_stage1_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "decimal128/i128", "data": "synthetic",
            "q1_steps_per_hour": 3600.0 / (ms / 1e3 / args.steps),
            "config": {"workload": "TPC-H q1 SF10 (BASELINE.json configs[1]): lineitem 59,986,052 rows x 7 columns, "
                                   "Arrow layout resident in HBM, 1 GPU executor per GPU", "rows_per_gpu": ROWS_SF10,
                       "target_partitions": P, "l2_policy": "inputs (4.68 GB per GPU) far larger than the 126 MB L2",
                       "stages": "scan+filter+project+partial-agg+hash-shuffle | final-agg+sort | merge",
                       "exchange": "in-library NCCL send/recv (b200_exchange_stage): hash repartition + gather to the merge task" if world > 1 else "none (1 executor)"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "fused_kernel<G=4,R=4,BT=256,shape=q1 with pre-packed key images> (stage 1: scan+filter+project+partial aggregate)",
                         "peak_source": peak_src, "kernel_ms": kern_s * 1e3, "algorithmic_bytes": alg_bytes},
            "gpu_launches": launches, "clocks": clocks,
            "parity_checked": bool(parity.get("checked") and parity.get("equal")), "parity": parity,
        }
        if world > 1:
            line["exchange"] = {"calls_per_step": exch_timed["calls"] / args.steps, "sent_bytes_per_step_rank0": exch_timed["sent"] / args.steps,
                                "recv_bytes_per_step_rank0": exch_timed["recv"] / args.steps}
        if e2e:
            line["e2e"] = e2e
        # CPU baseline beside it (rank 0): bounded sample of the same workload, on every CPU this process started with
        # (creating the engine bound this thread to the GPU's NUMA node)
        if not args.no_cpu_baseline:
            try:
                os.sched_setaffinity(0, START_AFFINITY)
            except Exception:
                pass
            threads = usable_cpus()
            rows = ROWS_SF10 // 4
            t, _ = cpu_q1(SF10_MSF, 0, rows, threads, steps=2, warmup=1)
            line["cpu_baseline"] = {"value": rows * len(t) / sum(t), "unit": "rows/s", "cores": threads, "kind": "port",
                                    "sample": f"q1 over {rows} lineitem rows (SF2.5), {threads} threads, 2 timed passes", "note": PORT_NOTE}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()
    if rank == 0 and parity.get("checked") and not parity.get("equal"):
        raise SystemExit(3)


# ---- other workloads: any TPC-H query (or all of them) under the distributed stage driver ---------------------
def run_workload(args):
    """Strong scaling: the tables of SF `--sf` are row-range partitioned over the N GPUs (dimension tables replicated),
    every stage is gang-scheduled and followed by the in-library exchange.  Reports base rows scanned / s, per-stage
    exchange bytes and, per kernel family, achieved GB/s on algorithmic bytes next to the measured HBM peak."""
    torch, dist, bb, eng, stream, device, rank, world, local_rank = setup_engine(args)
    import pyarrow as pa
    from ballista_b200 import tpch, driver
    fused = world > 1 and eng.counter("exchange_window_bytes") > 0
    names = sorted(tpch.QUERIES, key=lambda q: int(q[1:])) if args.workload == "all" else [args.workload]
    for nme in names:
        if nme not in tpch.QUERIES:
            raise SystemExit(f"unknown workload {nme}; have {sorted(tpch.QUERIES)}")
    sf = args.sf or {"q5": 25.0 * world, "q17": 12.5 * world}.get(args.workload, 10.0 * world)
    sf = min(sf, 100.0)
    msf = int(round(sf * 1000))
    P = world * max(1, args.partitions_per_gpu)

    def load(m):
        tabs = tpch.union_tables(names)
        tpch.TABLE_LAYOUT.clear()
        if len(names) > 1:
            tpch.TABLE_LAYOUT.update(tabs)
        # input partitions per GPU: as asked, but never more than ~120 M lineitem rows in one (Arrow Utf8 offsets are int32:
        # a partition's o_comment / l_comment characters must stay below 2 GiB)
        li_rows = 6_000_000 * m // 1000 // world
        in_parts = max(1, args.partitions_per_gpu, -(-li_rows // 120_000_000))
        return tabs, eng.tpch_load(tabs, m, rank, world, in_parts)

    def plans(PP):
        return {nme: tpch.QUERIES[nme][1](PP) for nme in names}

    # ---- parity first (untimed): the same distributed path at a scale the CPU oracle finishes in seconds ----------
    parity = {"checked": False}
    if not args.no_parity:
        pmsf = min(msf, 1000)
        tabs, _ = load(pmsf)
        pl = plans(P)
        got = {}
        for nme in names:
            got[nme] = driver.run_stages_distributed(eng, pl[nme], f"par-{nme}", rank, world, fused=fused)
            eng.synchronize()
            eng.remove_job_data(f"par-{nme}")
        if rank == 0:
            import oracle_ffi
            o = oracle_ffi.OracleEngine()
            for t, cols in tabs.items():
                n = eng.tpch_table_rows(t, pmsf)
                o.tpch_generate(t, pmsf, 0, 0, n, cols)
            bad = []
            t0 = time.perf_counter()
            for nme in names:
                want = driver.run_stages(o, pl[nme], f"o-{nme}")
                ordered = nme not in ("q3", "q10", "q18")   # top-k queries: ties beyond the sort keys
                g, w = got[nme], want
                if not ordered:
                    from util import canon
                    g, w = canon(g), canon(w)
                if not tables_equal(g, w, f64_rtol=1e-12):
                    bad.append(nme)
            o.close()
            parity = {"checked": True, "equal": not bad, "mismatch": bad, "oracle_seconds": time.perf_counter() - t0,
                      "what": f"{len(names)} queries through the same N={world} path at SF{pmsf / 1000:g} == CPU oracle (decimals/ints/strings bit-exact, f64 1e-12)"}
    tabs, rows_of = load(msf)
    pl = plans(P)
    eng.set_config("b200.metrics.kernel_timing", "on")

    exch = {}
    def on_stage(q):
        def cb(stage_id, mode, st):
            e = exch.setdefault(q, {"sent": 0, "recv": 0, "calls": 0, "max_sent_stage": 0})
            e["sent"] += st["sent_bytes"]
            e["recv"] += st["recv_bytes"]
            e["calls"] += 1
            e["max_sent_stage"] = max(e["max_sent_stage"], st["sent_bytes"])
        return cb

    def step(tag, timed):
        per_q = {}
        res = {}
        for nme in names:
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            res[nme] = driver.run_stages_distributed(eng, pl[nme], f"{tag}-{nme}", rank, world, on_stage=on_stage(nme) if timed else None, fused=fused)
            eng.synchronize()
            dt = time.perf_counter() - t0
            eng.remove_job_data(f"{tag}-{nme}")
            per_q[nme] = dt
        return per_q, res

    for w in range(max(args.warmup, 1)):
        step(f"warm{w}", False)
    eng.kernel_stats(reset=True)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = eng.kernel_launches()
    fused0 = eng.counter("fused_exchanges")
    acc = {nme: 0.0 for nme in names}
    res = None
    for k in range(args.steps):
        per_q, res = step(f"s{k}", True)
        # a query's time = the slowest rank's wall clock between two barriers
        t = torch.tensor([per_q[nme] for nme in names], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        for nme, v in zip(names, t.tolist()):
            acc[nme] += v
    clocks = sampler.stop() if rank == 0 else None
    launches = eng.kernel_launches() - launches0
    kstats = eng.kernel_stats(reset=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res)
    # self-consistency at full scale (the oracle cannot hold SF100): a different shuffle fan-out must give the same table
    consistent = None
    if not args.no_parity:
        pl2 = plans(P * 2)
        res2 = {}
        for nme in names:
            res2[nme] = driver.run_stages_distributed(eng, pl2[nme], f"alt-{nme}", rank, world, fused=fused)
            eng.synchronize()
            eng.remove_job_data(f"alt-{nme}")
        if rank == 0:
            from util import canon
            consistent = all(tables_equal(canon(res[nme]), canon(res2[nme]), f64_rtol=1e-12) for nme in names)
    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        sec = {nme: acc[nme] / args.steps for nme in names}
        total_s = sum(sec.values())
        rows = sum(tpch.base_rows(nme, rows_of) for nme in names)
        kern = {}
        for kname, st in sorted(kstats.items(), key=lambda kv: -kv[1]["ms"]):
            if st["launches"] == 0:
                continue
            gbs = st["bytes"] / (st["ms"] / 1e3) / 1e9 if st["ms"] > 0 else 0.0
            kern[kname] = {"ms_per_step": st["ms"] / args.steps, "launches_per_step": st["launches"] / args.steps,
                           "algorithmic_gb_per_step": st["bytes"] / args.steps / 1e9, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak}
        dom = next(iter(kern.items())) if kern else (None, None)
        line = {
            "metric": "tpch_rows_per_sec", "value": rows / total_s, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * total_s, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "decimal128/i128 (+f64 where the SQL forces it)", "data": "synthetic",
            "config": {"workload": f"TPC-H {args.workload} SF{sf:g}, {world} GPU executors, hash joins (prefer_hash_join=true), "
                                   f"target_partitions={P}, tables resident in HBM (row-range partitioned, nation/region replicated)",
                       "queries": names, "l2_policy": "inputs far larger than the 126 MB L2", "timing": "per query: max over ranks of the wall clock between barriers (device synchronised)"},
            "per_query_ms": {nme: 1e3 * sec[nme] for nme in names},
            "queries_per_hour": len(names) * 3600.0 / total_s,
            "base_rows_scanned": rows,
            "exchange_rank0": {q: {"calls": e["calls"] / args.steps, "sent_gb": e["sent"] / args.steps / 1e9, "recv_gb": e["recv"] / args.steps / 1e9,
                                   "largest_stage_sent_gb": e["max_sent_stage"] / 1e9} for q, e in exch.items()},
            "fused_shuffle": ({"window_gb": eng.counter("exchange_window_bytes") / (1 << 30), "exchanges_per_step": (eng.counter("fused_exchanges") - fused0) / args.steps,
                               "what": "writer + hash exchange as one collective: the scatter kernel stores rows into the owner's HBM over NVLink (fixed-width shuffles)"}
                              if fused else None),
            "kernels": kern,
            "roofline": ({"bound": "hbm", "kernel": dom[0], "achieved": dom[1]["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": dom[1]["frac_of_hbm_peak"],
                          "traffic": None, "peak_source": peak_src, "note": "dominant kernel family by device time; algorithmic bytes per SURVEY.md 8(d)"} if dom[0] else None),
            "gpu_launches": launches, "clocks": clocks,
            "parity_checked": bool(parity.get("checked") and parity.get("equal")), "parity": parity, "self_consistent_at_full_scale": consistent,
        }
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()
    if rank == 0 and ((parity.get("checked") and not parity.get("equal")) or consistent is False):
        raise SystemExit(3)


def measure_e2e(eng, bb, pa, torch, dist, step, rank, world, device, steps):
    """Same q1, but every step starts from HOST Arrow buffers (pinned) handed to the C-ABI
    (b200_engine_register_batch: H2D inside the timed region) and ends with the result on the host.
    At N > 1 every rank ingests its own share; the time is the max over ranks of the wall clock between barriers."""
    L = bb.engine.load_library()
    host = eng.export_table("lineitem", 0)  # device -> pageable host (setup, untimed)
    n = host.num_rows
    pinned, arrays, h2d = [], [], 0
    for col in host.columns:
        bufs = []
        for b in col.buffers():
            if b is None:
                bufs.append(None)
                continue
            p = L.b200_host_alloc_pinned(b.size + 64)
            if not p:
                raise RuntimeError("pinned allocation failed")
            C.memmove(p, b.address, b.size)
            pinned.append(p)
            bufs.append(pa.foreign_buffer(p, b.size))
            h2d += b.size
        arrays.append(pa.Array.from_buffers(col.type, n, bufs))
    batch = pa.RecordBatch.from_arrays(arrays, schema=host.schema)
    del host
    times = []
    d2h = 0
    saved0 = eng.counter("ingest_bytes_saved")
    for k in range(steps + 1):
        job = f"e2e#{k}"
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        eng.drop_table("lineitem_host")
        eng.register_batch("lineitem_host", 0, batch)
        res = step(job, table="lineitem_host")
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        if res is not None:
            d2h = res.nbytes
        if k > 0:
            times.append(dt)
    eng.drop_table("lineitem_host")
    for p in pinned:
        L.b200_host_free_pinned(p)
    # bytes that actually crossed PCIe: Decimal128 columns whose values fit 32/64 bits are narrowed by the
    # engine's host pool before the copy and widened back on the device (bit-exact; csrc/host/host_pool.hpp)
    saved = (eng.counter("ingest_bytes_saved") - saved0) // (steps + 1)
    return {"value": n * world * len(times) / sum(times), "unit": "rows/s", "h2d_bytes_per_step": (h2d - saved) * world, "d2h_bytes_per_step": d2h,
            "ms_per_step": 1e3 * sum(times) / len(times), "steps": len(times), "host_arrow_bytes_per_step": h2d * world,
            "note": "host pinned Arrow buffers (host_arrow_bytes_per_step) -> b200_engine_register_batch (host pool narrows "
                    "Decimal128 sign-extension bytes, H2D of h2d_bytes_per_step, device widens) -> 3 stages (+ exchanges) -> b200_partition_export (D2H)"}


DUMP_LIMIT_BYTES = 64 << 20


def _column_to_numpy(col):
    """One result column as float64 (nulls NaN); a string column as a float32 [rows, longest] matrix of its UTF-8 bytes,
    zero-padded, a null row all NaN."""
    import numpy as np
    import pyarrow as pa
    t = col.type
    if pa.types.is_string(t) or pa.types.is_large_string(t) or pa.types.is_binary(t):
        vals = [None if v is None else (v.encode() if isinstance(v, str) else v) for v in col.to_pylist()]
        out = np.zeros((len(vals), max([1] + [len(v) for v in vals if v is not None])), np.float32)
        for i, v in enumerate(vals):
            if v is None:
                out[i] = np.nan
            else:
                out[i, :len(v)] = np.frombuffer(v, np.uint8)
        return out
    if pa.types.is_date32(t):
        col = col.cast(pa.int32())
    elif pa.types.is_temporal(t):
        col = col.cast(pa.int64())
    return col.cast(pa.float64()).to_numpy(zero_copy_only=False).astype(np.float64)


def dump_outputs(out_dir, results):
    """results: {query: result table (pyarrow Table or RecordBatch) of the last timed step}.  Writes every column as
    out_dir/<query>_<column>.npy.  Past DUMP_LIMIT_BYTES in all, each table keeps the same seeded sample of its rows
    (in order) and its row numbers go to <query>__rows.npy."""
    import numpy as np
    import pyarrow as pa
    os.makedirs(out_dir, exist_ok=True)
    tables = {q: pa.Table.from_batches([r]) if isinstance(r, pa.RecordBatch) else r for q, r in results.items() if r is not None}
    arrays = {q: [(name, _column_to_numpy(t.column(name))) for name in t.column_names] for q, t in tables.items()}
    per_table = (DUMP_LIMIT_BYTES - (1 << 20)) // max(1, len(arrays))     # 1 MB left for the .npy headers
    for q, cols in arrays.items():
        n = tables[q].num_rows
        row_bytes = sum(a.nbytes // max(1, n) for _, a in cols)
        keep = n if row_bytes * n <= per_table else per_table // (row_bytes + 8)
        if keep < n:
            rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
            np.save(os.path.join(out_dir, f"{q}__rows.npy"), rows.astype(np.float64))
            cols = [(name, a[rows]) for name, a in cols]
        for name, a in cols:
            np.save(os.path.join(out_dir, f"{q}_{name}.npy"), a)
    log(f"dumped {sum(len(c) for c in arrays.values())} result columns of {sorted(arrays)} to {out_dir}")


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line goes to the process' real stdout; everything else a library prints there (NCCL's version banner,
    torchrun notices) was redirected to stderr when the run started."""
    txt = json.dumps(line) + "\n"
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, txt.encode())
    else:
        sys.stdout.write(txt)
        sys.stdout.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="q1", help="q1 (headline, weak scaling) | q5 | q17 | all | any TPC-H query name (strong scaling at --sf)")
    ap.add_argument("--sf", type=float, default=0.0, help="scale factor of the non-q1 workloads (default: chosen per workload and N)")
    ap.add_argument("--partitions-per-gpu", type=int, default=1)
    ap.add_argument("--exchange-window-gb", type=float, default=-1.0, help="HBM per executor for the fused shuffle (N>1; default 16 for the non-q1 workloads)")
    ap.add_argument("--no-fused-shuffle", action="store_true", help="N>1: always shuffle in two steps (writer, then NCCL exchange)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the result of the last one as DIR/<query>_<column>.npy "
                                                          "(float64; strings as float32 byte matrices; at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
