#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for the VisionLLMv2 forward hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--dump-outputs DIR]

One JSON line on rank 0.  See DESIGN.md "Measurement" for what each field means.
With --dump-outputs, rank 0 also writes the arrays its last timed step returned to DIR/<name>.npy (see dump_outputs),
so that two builds can be compared output for output on the same seeded inputs.  It needs --impl native: the reference
arm times a bounded CPU sample of the path (one layer per tower), not the path's outputs.
Workloads live in bench_workloads.py; the default is the most complete
native path available (see DEFAULT_WORKLOAD there).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.rows = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6),
                              ("sw_power_cap", 7)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


_T0 = time.time()


def trace(msg):
    """Stage timestamps on stderr (VLLM_BENCH_TRACE=1): where a multi-rank launch spends its start-up time."""
    if os.environ.get("VLLM_BENCH_TRACE"):
        print(f"[bench rank {os.environ.get('RANK', '0')} +{time.time() - _T0:6.1f}s] {msg}", file=sys.stderr, flush=True)


DUMP_BUDGET_BYTES = 64 * 10 ** 6
NPY_HEADER_BYTES = 128                     # numpy writes a 128-byte header for these 1-D / few-dim arrays


def dump_outputs(out, directory, budget=DUMP_BUDGET_BYTES):
    """Write every tensor in one step's result (nested dicts / lists / tuples, e.g. a ModelOutput) as
    `directory/<dotted name>.npy`: floating types other than float64 become float32; float64 and integer types become
    float64 (exact for integers below 2^53).  When that would take more than `budget` bytes, each array is replaced by
    a sample of its flattened elements -- distinct indices drawn by a generator seeded with 0, sorted, a share of the
    budget proportional to the array's size, at least one element -- and the indices are written as float64 to
    `directory/sample_index/<dotted name>.npy`.  The budget counts whole files, headers included.  The same elements are written on every run
    with the same arguments.  Returns {name: {"shape", "dtype", "elements_written"}}."""
    import numpy as np
    import torch
    arrays = {}

    def walk(name, x):
        if isinstance(x, torch.Tensor):
            arrays[name or "out"] = x.detach()
        elif isinstance(x, dict):
            for k, v in x.items():
                walk(f"{name}.{k}" if name else str(k), v)
        elif isinstance(x, (list, tuple)):
            for i, v in enumerate(x):
                walk(f"{name}.{i}" if name else str(i), v)

    walk("", out)
    if not arrays:
        raise RuntimeError(f"--dump-outputs: the step returned no tensors ({type(out).__name__})")
    wide = {n: t.dtype == torch.float64 or not (t.is_floating_point() or t.dtype == torch.bool) for n, t in arrays.items()}
    width = {n: 8 if wide[n] else 4 for n in arrays}
    sampled = sum(t.numel() * width[n] + NPY_HEADER_BYTES for n, t in arrays.items()) > budget
    if sampled:
        cost = sum(t.numel() * (width[n] + 8) for n, t in arrays.items())     # value + float64 index per element
        room = budget - (16 + 2 * NPY_HEADER_BYTES) * len(arrays)            # headers, at-least-one-element guarantee
        os.makedirs(os.path.join(directory, "sample_index"), exist_ok=True)
    os.makedirs(directory, exist_ok=True)
    manifest = {}
    for name, t in arrays.items():
        flat = t.reshape(-1)
        if sampled and flat.numel():
            keep = min(flat.numel(), max(1, flat.numel() * room // cost))
            g = torch.Generator(device=flat.device).manual_seed(0)
            idx = torch.randperm(flat.numel(), generator=g, device=flat.device)[:keep].sort().values
            flat = flat[idx]
            np.save(os.path.join(directory, "sample_index", name + ".npy"), idx.to(torch.float64).cpu().numpy())
        a = flat.to(torch.float64 if wide[name] else torch.float32).cpu().numpy()
        np.save(os.path.join(directory, name + ".npy"), a if sampled else a.reshape(tuple(t.shape)))
        manifest[name] = {"shape": list(t.shape), "dtype": str(t.dtype).replace("torch.", ""), "elements_written": a.size}
    return manifest


_REAL_STDOUT = None


def quiet_stdout():
    """Libraries print to fd 1 (NCCL's "NCCL version ..." banner at communicator creation): park the real stdout and
    send everything else to stderr, so that the ONE JSON line is the only thing on stdout."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (each timed loop runs exactly this many)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cuprof", action="store_true",
                    help="wrap ONE extra device step in cudaProfilerStart/Stop (ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs needs --impl native (the reference arm times a CPU sample, not the path's outputs)")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else max(args.warmup, 1)

    import bench_workloads as benchlib
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    name = args.workload or benchlib.DEFAULT_WORKLOAD

    if args.impl == "reference":
        # The reference's CPU implementation of the path, on the host cores; rank 0 only.
        if rank != 0:
            return
        line = benchlib.run_reference_arm(name, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup)
        print(json.dumps(line), flush=True)
        return

    quiet_stdout()
    trace("importing torch")
    import torch
    import torch.distributed as dist
    trace("torch imported")
    torch.cuda.set_device(local_rank)
    torch.cuda.init()
    trace("cuda context up")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        trace("process group up")
    wl = benchlib.WORKLOADS[name](rank=rank, world=world, device=torch.device("cuda", local_rank))
    wl.setup()
    trace("workload set up")

    from visionllm_b200 import _lib

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        """EXACTLY `steps` calls, barrier+sync on both sides, CUDA events, max over ranks -> ms total."""
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        launches = _lib.launch_count() - l0
        barrier()
        return benchlib.max_over_ranks(e0.elapsed_time(e1), dist if world > 1 else None, "cuda"), launches

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev, launches = timed(wl.step_device, args.steps, args.warmup)
    trace(f"device-resident steps timed: {ms_dev / args.steps:.2f} ms/step")
    dumped = dump_outputs(wl.out, args.dump_outputs) if args.dump_outputs and rank == 0 else None
    if args.cuprof:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        wl.step_device()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    kern = wl.dominant_kernel_ms(args.steps)            # live CUDA-event time of the dominant kernel
    ms_e2e, _ = timed(wl.step_e2e, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else None
    tp_obj = None
    if world > 1 and name == benchlib.DEFAULT_WORKLOAD and not os.environ.get("VLLM_BENCH_NO_EXTRAS"):
        try:                                               # cfg 5 under the same launch (all ranks take part)
            tp_obj = benchlib.tp_extra(rank, world, torch.device("cuda", local_rank))
        except Exception as e:
            tp_obj = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    units = wl.units_per_step() * world
    peaks = benchlib.measured_peaks()
    roof = wl.roofline(kern, peaks)
    line = {
        "metric": wl.metric, "value": units / (ms_dev / args.steps / 1e3), "unit": wl.unit,
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": wl.dtype,
        "data": "synthetic", "config": wl.config(),
        "e2e": {"value": units / (ms_e2e / args.steps / 1e3), "unit": wl.unit,
                "h2d_bytes_per_step": wl.h2d_bytes, "d2h_bytes_per_step": wl.d2h_bytes,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches, "clocks": clocks, "roofline": roof,
    }
    line.update(wl.extra())
    if tp_obj is not None:
        line["tp"] = tp_obj
    if dumped is not None:
        line["dumped_outputs"] = {"dir": os.path.abspath(args.dump_outputs), "arrays": dumped}
    if name == benchlib.DEFAULT_WORKLOAD and not os.environ.get("VLLM_BENCH_NO_EXTRAS"):
        try:                                               # the "deform-attn HBM GB/s" half of BASELINE.json's metric
            line["msda"] = benchlib.msda_extra(torch.device("cuda", local_rank))
        except Exception as e:
            line["msda"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = benchlib.cpu_baseline(name)
    emit(line)
    if world > 1:
        os.dup2(2, 1)                                  # teardown chatter stays off stdout too
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
