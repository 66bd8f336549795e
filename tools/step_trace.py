"""Device timeline of resident-input q1 steps under torch.profiler (CUDA activities): for every step, each kernel, memcpy
and memset with its duration and the device idle gap before it, plus the engine's kernel launches and stream
synchronisations.  The call sequence is bench.py's step() at N=1 (prepare + execute stages 1..3, export, drop the job).
Tracing slows the host, so the gaps are upper bounds of the untraced ones; take step times from bench.py, not from here.

    python tools/step_trace.py [--msf 10000] [--steps 20] [--warmup 3] [--out FILE]"""
import argparse
import json
import os
import statistics
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--msf", type=int, default=10000, help="scale factor x 1000 of the lineitem table (10000 = SF10)")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="write the report here as well as to stdout")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile, record_function
    import ballista_b200 as bb
    from ballista_b200 import tpch

    if not torch.cuda.is_available():
        raise SystemExit("step_trace needs a GPU")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    eng = bb.GpuExecutionEngine(0)
    stream = torch.cuda.Stream(device=dev)
    eng.set_stream(stream.cuda_stream)
    n = eng.tpch_table_rows("lineitem", args.msf)
    eng.tpch_generate("lineitem", args.msf, 0, 0, n, tpch.Q1_COLUMNS)
    stages = tpch.q1(n_partitions=1)

    def step(job):
        for st in stages:
            s = eng.create_query_stage_exec(job, st.stage_id, st.json(job))
            s.execute_query_stage(0)
            s.release()
        out = eng.partition_export(job, 3, 0)
        eng.remove_job_data(job)
        return out

    for w in range(max(args.warmup, 3)):
        step(f"warm#{w}")
    torch.cuda.synchronize(dev)

    counts = []
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for k in range(args.steps):
            l0, s0 = eng.kernel_launches(), eng.counter("stream_syncs")
            with record_function(f"q1_step#{k}"):
                step(f"trace#{k}")
            counts.append((eng.kernel_launches() - l0, eng.counter("stream_syncs") - s0))
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    eng.close()

    evs = [e for e in trace.get("traceEvents", []) if e.get("ph") == "X"]
    steps = sorted((e for e in evs if e.get("cat") == "user_annotation" and e.get("name", "").startswith("q1_step#")), key=lambda e: e["ts"])
    dev_ops = sorted((e for e in evs if e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")), key=lambda e: e["ts"])
    host_syncs = [e for e in evs if e.get("cat") == "cuda_runtime" and e.get("name") in ("cudaStreamSynchronize", "cudaDeviceSynchronize")]

    lines = []
    out = lines.append
    props = torch.cuda.get_device_properties(dev)
    out(f"# q1 step trace: lineitem msf={args.msf} ({n} rows), {args.steps} traced steps after {max(args.warmup, 3)} warm-up steps")
    out(f"# device: {props.name}; times in microseconds from torch.profiler (CUDA activities); gap = device idle before the op")
    summary = []
    for k, s in enumerate(steps):
        t0, t1 = s["ts"], s["ts"] + s["dur"]
        ops = [e for e in dev_ops if t0 <= e["ts"] < t1]
        n_sync = sum(1 for e in host_syncs if t0 <= e["ts"] < t1)
        busy = sum(e["dur"] for e in ops)
        out(f"step {k}: host {s['dur']:.1f} us, device busy {busy:.1f} us, {len(ops)} device ops, engine counters: "
            f"kernel_launches {counts[k][0]}, stream_syncs {counts[k][1]}; cudaStreamSynchronize calls {n_sync}")
        prev = t0
        for e in ops:
            gap = e["ts"] - prev
            kind = {"kernel": "kernel", "gpu_memcpy": "memcpy", "gpu_memset": "memset"}[e["cat"]]
            out(f"  {kind:6s} {e['dur']:9.1f}  gap {gap:8.1f}  {e['name'][:110]}")
            prev = max(prev, e["ts"] + e["dur"])
        tail = t1 - prev
        out(f"  tail after the last device op: {tail:.1f}")
        summary.append((s["dur"], busy, s["dur"] - busy, len(ops), n_sync, counts[k][0], counts[k][1]))
    if summary:
        med = [statistics.median(c) for c in zip(*summary)]
        out(f"median over {len(summary)} steps: host {med[0]:.1f} us, device busy {med[1]:.1f} us, device idle {med[2]:.1f} us, device ops {med[3]:g}, "
            f"cudaStreamSynchronize {med[4]:g}, kernel_launches {med[5]:g}, stream_syncs {med[6]:g}")
    txt = "\n".join(lines) + "\n"
    sys.stdout.write(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
