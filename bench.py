#!/usr/bin/env python
"""bench.py -- batched complex-FFT GFLOP/s (5 N log2 N) on B200 vs the HBM roofline.

Workload (BASELINE.json configs[1]): f32 forward, N = 2^10 .. 2^20, batch = 4096 per GPU, synthetic
U[0,10) complex vectors.  One "step" = one pass of the hot path over that whole sweep (11 sizes).

  python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's CUDA path
  python bench.py --impl reference ...                          # the reference's CPU path (see below)
  torchrun --nproc-per-node N ... bench.py --gpus N ...         # one rank per GPU, weak scaling

value   : whole-job GFLOP/s, inputs resident in HBM, CUDA events on the launch stream, max over ranks
e2e     : same metric through the host-slice C ABI (b200fft_exec_host_outofplace) from pinned host
          memory -- H2D and D2H inside the timed region (PCIe bound)
roofline: algorithmic bytes (read + write of the signal = 16 N per f32 transform, SURVEY.md 8(d)) /
          device time, against MEASURED_PEAKS.json hbm_gbs; per size and for the whole step
cpu_baseline / --impl reference: RustFFT itself cannot be built here (no rustc/cargo in the image), so
          the reference arm is the C++ restatement of its scalar planner path (oracle/, kind "port")
          on all host cores, one contiguous batch slice per thread (examples/concurrency.rs), on a
          bounded sample of the same sweep.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

LOGS = list(range(10, 21))
BATCH = 4096
METRIC = "batched complex-FFT GFLOP/s (5N log2 N), f32 forward, N=2^10..2^20, batch=4096/GPU"


def flops(n: int, batch: int) -> float:
    return 5.0 * n * math.log2(n) * batch


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
def host_threads() -> int:
    """CPUs this process may really use: the affinity mask, capped by the cgroup CPU quota (a container that shows 128 CPUs but is
    throttled to ~10 runs 128 spinning workers slower than 10)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        n = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota:
        n = max(1, min(n, int(math.ceil(quota))))
    return n


_cpu_buf = None


def cpu_sample(threads: int, min_reps: int = 5, target_s: float = 0.25, logs=None):
    """One pass of the SAME workload on the host: every N in 2^10..2^20 with batch = 4096 (BASELINE configs[1]), in place, f32,
    through the C++ port of RustFFT's scalar planner path -- `threads` pinned workers created once per size outside the timed
    passes, each with its own contiguous slice of the batch (examples/concurrency.rs), >= `min_reps` separately timed passes per
    size (more for the small sizes, to ~target_s), median pass per size.  Returns (GFLOP/s of the sweep, seconds of timed CPU
    work, per-size rows).  Sizes whose single pass already takes >= target_s are timed once (after no extra warm-up pass: the
    first touch of the buffer happens before the timed region inside oracle_bench_f32)."""
    import numpy as np

    import oracle

    global _cpu_buf
    logs = logs or LOGS
    batch = BATCH
    if _cpu_buf is None:
        while True:
            try:
                _cpu_buf = np.empty(batch << max(logs), dtype=np.complex64)  # untouched pages: the workers first-touch their slices
                break
            except MemoryError:  # pragma: no cover  (a box without 32 GiB to spare: shrink the batch and say so)
                batch //= 2
    batch = _cpu_buf.size >> max(logs)
    total_f, total_t, spent, per = 0.0, 0.0, 0.0, []
    for lg in logs:
        n = 1 << lg
        f = flops(n, batch)
        first = oracle.bench_f32(n, batch, threads, 1, _cpu_buf)[0]  # one pass: warms this size up and sizes the sample
        spent += first
        if first >= target_s:
            ts = [first]  # a pass of this size already is a bounded sample (seconds of work on every thread)
        else:
            ts = sorted(oracle.bench_f32(n, batch, threads, int(min(200, max(min_reps, math.ceil(target_s / max(first, 1e-6))))), _cpu_buf))
        reps = len(ts)
        med = ts[len(ts) // 2]
        per.append({"log2n": lg, "batch": batch, "reps": reps, "gflops": round(f / med / 1e9, 2), "gflops_best": round(f / ts[0] / 1e9, 2),
                    "gflops_per_core": round(f / med / 1e9 / threads, 3)})
        total_f += f
        total_t += med
        spent += sum(ts)
    return total_f / total_t / 1e9, spent, per


def scipy_sample(threads: int, logs=None):
    """Second CPU comparator (NOT RustFFT): scipy.fft (pocketfft, SIMD over the batch) with workers = all host threads, complex64,
    batch = min(4096, 2^27 / N) transforms per size, best of 3."""
    try:
        import numpy as np
        import scipy.fft as sfft
    except Exception as e:  # pragma: no cover
        return {"error": f"{type(e).__name__}: {e}"[:120]}
    logs = logs or LOGS
    rng = np.random.default_rng(7)
    total_f, total_t, per = 0.0, 0.0, []
    for lg in logs:
        n = 1 << lg
        batch = max(1, min(BATCH, (1 << 27) // n))
        x = (rng.random((batch, n), dtype=np.float32) + 1j * rng.random((batch, n), dtype=np.float32)).astype(np.complex64)
        best = 1e30
        for _ in range(3):
            t0 = time.perf_counter()
            sfft.fft(x, axis=-1, workers=threads)
            best = min(best, time.perf_counter() - t0)
        f = flops(n, batch)
        per.append({"log2n": lg, "batch": batch, "gflops": round(f / best / 1e9, 2)})
        total_f += f
        total_t += best
    return {"value": round(total_f / total_t / 1e9, 2), "unit": "GFLOP/s", "workers": threads, "what": "scipy.fft.fft complex64 (pocketfft), "
            "batch = min(4096, 2^27/N) per size, best of 3 -- a vectorised CPU FFT, not RustFFT", "per_size": per}


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    import oracle

    oracle.build()
    cores = host_threads()
    logs = LOGS if not args.logs else [int(x) for x in args.logs.split(",")]
    if args.warmup:  # ONE light untimed pass (small sizes only) warms the code; every size's timed sample warms its own data
        cpu_sample(cores, min_reps=2, target_s=0.0, logs=[lg for lg in logs if lg <= 14] or logs[:1])
    vals, t_all, per = [], 0.0, None
    for _ in range(args.steps):
        g, t, per = cpu_sample(cores, logs=logs)
        vals.append(g)
        t_all += t
    value = sorted(vals)[len(vals) // 2]
    step_ms = 1e3 * sum(flops(1 << lg, per[0]["batch"]) for lg in logs) / (value * 1e9)
    sample = (f"per step: every N in 2^10..2^20 with batch = {per[0]['batch']} (the GPU arm's workload), in place; sizes whose pass is shorter than 0.25 s "
              "are timed >= 5 times (median pass), longer ones once; workers created and pinned once per size outside the timed passes; "
              f"threads = {cores} = CPUs usable by this process (affinity mask capped by the cgroup quota)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(value, 2), "unit": "GFLOP/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(step_ms, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE configs[1]: f32 forward, N=2^10..2^20, batch=4096 per GPU, out of place, "
                               "device resident", "sizes_log2": logs, "batch_per_gpu": BATCH,
                   "reference_arm": "C++ port of RustFFT's scalar planner path (oracle/; RustFFT itself needs rustc, absent from the image), "
                                    "in place on host memory, all host threads", "per_size": per},
        "cpu_baseline": {"value": round(value, 2), "unit": "GFLOP/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 2), "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "scipy_fft": scipy_sample(cores, logs),
    }), flush=True)


# ------------------------------------------------------------------------------------------
class NvmlSampler:
    """SM clock + throttle reasons through NVML every ~5 ms (nvidia-smi -lms 100 yields only 1-3 lines inside a
    0.2 s timed region).  Entirely optional: any failure leaves `result()` None and the nvidia-smi sampler is used."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, index: int, nvml=None):
        self.ok, self.samples, self.mask, self.mx, self.stop_flag, self.thread = False, [], 0, None, False, None
        try:
            if nvml is None:
                import pynvml as nvml
            self.nvml = nvml
            nvml.nvmlInit()
            self.h = nvml.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(nvml.nvmlDeviceGetMaxClockInfo(self.h, nvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            self.ok = False

    def _loop(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                self.mask |= int(get(self.h))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if not self.ok:
            return
        try:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception:
            self.ok = False

    def result(self):
        try:
            self.stop_flag = True
            if self.thread:
                self.thread.join(timeout=1)
            if not self.ok or len(self.samples) < 3:
                return None
            sm = sorted(self.samples)
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.mx, "reasons": sorted(n for b, n in self.REASONS if self.mask & b),
                    "samples": len(sm), "source": "nvml"}
        except Exception:
            return None


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.nvml = NvmlSampler(index)

    def start(self):
        self.nvml.start()
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        fast = self.nvml.result()
        if fast is not None:
            if self.proc:
                try:
                    self.proc.terminate()
                    self.proc.wait(timeout=2)
                except Exception:
                    pass
            return fast
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def bind_to_gpu_numa_node(index: int):
    """Multi-GPU runs: keep this rank's host threads (and therefore the first touch of its pinned buffers and the copy pool of the
    host-slice path) on the NUMA node its GPU hangs off -- round 1's 8-GPU e2e run lost 39 % to ranks copying across sockets.
    Returns a short description for the bench line, or None when the topology cannot be read (then nothing is changed)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:  # NVML prints an 8-digit domain, sysfs uses 4
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return f"node{node}:{len(cpus)}cpus"
    except Exception:
        return None


def run_ours(args, rank: int, world: int, local_rank: int):
    import numpy as np
    import torch

    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None

    import rustfft_b200 as rb

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)

    planner = rb.FftPlanner(np.complex64, device=local_rank)
    plans = {lg: planner.plan_fft_forward(1 << lg) for lg in LOGS}
    logs = LOGS if not args.logs else [int(x) for x in args.logs.split(",")]

    # one 32 GiB input region + one 32 GiB output region; sizes below 2^20 live at disjoint offsets so
    # nothing a size reads was touched since >= 32 GiB of other traffic (no L2 reuse between sizes/steps)
    max_elems = BATCH << max(logs)
    offs, o = {}, 0
    for lg in logs:
        if lg == max(logs):
            offs[lg] = 0
        else:
            offs[lg] = o
            o += BATCH << lg
    src = torch.empty(max_elems, dtype=torch.complex64, device=dev)
    dst = torch.empty(max_elems, dtype=torch.complex64, device=dev)
    g = torch.Generator(device=dev).manual_seed(20260922 + rank)
    step_e = 1 << 26
    for i in range(0, max_elems, step_e):
        k = min(step_e, max_elems - i)
        torch.view_as_real(src[i:i + k]).copy_(torch.rand(k, 2, device=dev, generator=g) * 10)
    ws_bytes = max(plans[lg].workspace_bytes(BATCH) for lg in logs)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)

    def one_size(lg, rep=0):
        n = 1 << lg
        o = offs[lg] if rep == 0 else (rep * BATCH * n) % max_elems
        a = src[o: o + BATCH * n]
        b = dst[o: o + BATCH * n]
        plans[lg].process_device(a, out=b, workspace=ws if plans[lg].workspace_bytes(BATCH) else None)

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    n_warm = (0 if args.profile_cold else 1) if args.profile else max(args.warmup, 3)
    for _ in range(n_warm):
        for lg in logs:
            one_size(lg)
    barrier()

    # Launch path: each size's exec is captured once into a CUDA graph and replayed, so the GPU never
    # waits for the Python/ctypes launch path between kernels (the library issues up to ~1000 launches
    # per exec for the chunked two-pass plans).  Falls back to plain stream launches if capture fails.
    launch_mode = "cuda-graph replay (one graph per size)"
    graphs, rep_graphs, reps = {}, {}, {}
    if args.profile or args.no_graph:
        launch_mode = "stream launches"
    else:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for lg in logs:
                    g1 = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g1, stream=side):
                        one_size(lg)
                    graphs[lg] = g1
                    # supplementary per-size measurement: R back-to-back execs over R distinct regions (>= 2 GiB)
                    reps[lg] = max(1, min(64, (1 << 31) // (8 * (BATCH << lg))))
                    g2 = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g2, stream=side):
                        for r in range(reps[lg]):
                            one_size(lg, rep=r + 1 if reps[lg] > 1 else 0)
                    rep_graphs[lg] = g2
            torch.cuda.current_stream().wait_stream(side)
        except Exception as e:  # pragma: no cover
            launch_mode = f"stream launches (graph capture failed: {type(e).__name__})"
            graphs, rep_graphs = {}, {}

    def run_size(lg):
        if graphs:
            graphs[lg].replay()
        else:
            one_size(lg)

    if not args.profile:
        for lg in logs:  # one more warm-up through the final launch path
            run_size(lg)
    barrier()

    # --dump-outputs: the same seeded choice of whole transforms of every size in every run (2^19 elements per size, one
    # transform at 2^20: 48 MiB for the default sweep), taken from rank 0's last timed step
    dump_rows = {}
    if args.dump_outputs and rank == 0:
        pick = np.random.default_rng(1234)
        dump_rows = {lg: torch.from_numpy(np.sort(pick.choice(BATCH, max(1, (1 << 19) >> lg), replace=False))).to(dev) for lg in logs}
    dumped = {}

    sampler = ClockSampler(local_rank)
    sampler.start()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(len(logs) + 1)] for _ in range(args.steps)]
    begin = [row[:-1] for row in ev]  # size i of step s is timed from begin[s][i] to ev[s][i + 1]
    barrier()
    for s in range(args.steps):
        ev[s][0].record()
        for i, lg in enumerate(logs):
            run_size(lg)
            ev[s][i + 1].record()
            if dump_rows and s == args.steps - 1:
                # every size's output region lies inside the largest size's, so each output is sampled before the next size
                # runs; the next size's window starts after the copy, which stays out of the timing
                n = 1 << lg
                dumped[lg] = dst[offs[lg]: offs[lg] + BATCH * n].view(BATCH, n).index_select(0, dump_rows[lg])
                if i + 1 < len(logs):
                    begin[s][i + 1] = torch.cuda.Event(enable_timing=True)
                    begin[s][i + 1].record()
    barrier()
    clocks = sampler.stop()
    total_ms = ev[0][0].elapsed_time(ev[-1][-1])
    if dump_rows:
        total_ms -= sum(ev[-1][i].elapsed_time(begin[-1][i]) for i in range(1, len(logs)))
    per_ms = {lg: sum(begin[s][i].elapsed_time(ev[s][i + 1]) for s in range(args.steps)) / args.steps
              for i, lg in enumerate(logs)}
    if dumped:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for lg, rows in dumped.items():
            np.save(os.path.join(args.dump_outputs, f"fft_f32_forward_log2n{lg}.npy"), torch.view_as_real(rows).cpu().numpy())
    # supplementary: per-size time from R back-to-back execs (amortises the ~10 us launch+drain of a single
    # exec, which is comparable to the whole transform time at N = 2^10..2^12)
    per_ms_rep = {}
    if rep_graphs:
        for lg in logs:
            rep_graphs[lg].replay()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rep_graphs[lg].replay()
            e1.record()
            torch.cuda.synchronize()
            per_ms_rep[lg] = e0.elapsed_time(e1) / reps[lg]
    if dist:
        t = torch.tensor([total_ms] + [per_ms[lg] for lg in logs] + [per_ms_rep.get(lg, 0.0) for lg in logs],
                         device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = t[0].item()
        per_ms = {lg: t[i + 1].item() for i, lg in enumerate(logs)}
        if per_ms_rep:
            per_ms_rep = {lg: t[i + 1 + len(logs)].item() for i, lg in enumerate(logs)}

    hbm, peak_src = peaks()
    step_ms = total_ms / args.steps
    step_flops = sum(flops(1 << lg, BATCH) for lg in logs)
    step_bytes = sum(16.0 * (1 << lg) * BATCH for lg in logs)
    value = step_flops * world / (step_ms * 1e-3) / 1e9
    per_size = []
    for lg in logs:
        gbs = 16.0 * (1 << lg) * BATCH / (per_ms[lg] * 1e-3) / 1e9
        row = {"log2n": lg, "plan": plans[lg].describe(), "ms": round(per_ms[lg], 4),
               "gflops": round(flops(1 << lg, BATCH) / (per_ms[lg] * 1e-3) / 1e9, 1),
               "gbs": round(gbs, 1), "frac": round(gbs / hbm, 4)}
        if lg in per_ms_rep:
            g2 = 16.0 * (1 << lg) * BATCH / (per_ms_rep[lg] * 1e-3) / 1e9
            row.update({"back_to_back_reps": reps[lg], "ms_b2b": round(per_ms_rep[lg], 4), "gbs_b2b": round(g2, 1),
                        "frac_b2b": round(g2 / hbm, 4)})
        per_size.append(row)
    achieved = step_bytes / (step_ms * 1e-3) / 1e9
    dom = max(per_size, key=lambda r: r["ms"])  # the size (= kernel pair) the step spends most of its time in
    dominant = {"kernel": dom["plan"] + " at N=2^%d, batch %d (every launch of the plan, CUDA events around the exec)" % (dom["log2n"], BATCH),
                "share_of_step": round(dom["ms"] / step_ms, 3), "achieved": dom["gbs"], "frac": dom["frac"], "unit": "GB/s",
                "algorithmic_bytes_per_exec": int(16 * (1 << dom["log2n"]) * BATCH), "launches_per_exec": plans[dom["log2n"]].launches(BATCH)}
    launches = sum(plans[lg].launches(BATCH) for lg in logs) * args.steps
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("dram_bytes_per_step")

    # ---- e2e: the host-slice trait path (rank-local), PCIe inside the timing: pinned host buffers (headline) and pageable ones
    e2e = None
    if not args.no_e2e:
        cap = int(args.e2e_pinned_gib * (1 << 30)) // 8
        hin = torch.empty(min(cap, max_elems), dtype=torch.complex64).pin_memory()
        hout = torch.empty_like(hin).pin_memory()
        torch.view_as_real(hin).uniform_(0, 10)
        hin_np, hout_np = hin.numpy(), hout.numpy()

        def e2e_step(a_np, b_np):
            for lg in logs:
                n = 1 << lg
                todo = BATCH
                per_call = max(1, min(BATCH, a_np.size // n))
                while todo:
                    nb = min(per_call, todo)
                    plans[lg].process_outofplace_with_scratch(a_np[: nb * n], b_np[: nb * n])
                    todo -= nb

        def timed_e2e(a_np, b_np, steps):
            e2e_step(a_np, b_np)  # warm-up (pipeline resources, page faults)
            barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                e2e_step(a_np, b_np)
            barrier()
            sec = (time.perf_counter() - t0) / steps
            if dist:
                tt = torch.tensor([sec], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                sec = tt.item()
            return sec

        e2e_s = timed_e2e(hin_np, hout_np, args.e2e_steps)
        # the link itself: concurrent H2D + D2H of 1 GiB blocks on two streams (what any host pipeline is bounded by)
        blk = min(1 << 27, hin.numel())
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        dtmp = torch.empty(blk, dtype=torch.complex64, device=dev)
        dtmp2 = torch.empty(blk, dtype=torch.complex64, device=dev)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(4):
            with torch.cuda.stream(s1):
                dtmp.copy_(hin[:blk], non_blocking=True)
            with torch.cuda.stream(s2):
                hout[:blk].copy_(dtmp2, non_blocking=True)
        torch.cuda.synchronize()
        link = 4 * blk * 8 / (time.perf_counter() - t0) / 1e9
        del dtmp, dtmp2
        # pageable caller (what a Rust Vec is): staged through the library's pinned ring by its copy threads
        pg_in = np.empty(hin_np.size, dtype=np.complex64)
        pg_in[:] = hin_np
        pg_out = np.empty_like(pg_in)
        pg_s = timed_e2e(pg_in, pg_out, 1)
        del pg_in, pg_out
        # config 1's GPU twin: one N = 1024 transform through process() (H2D + kernel + D2H + sync), pageable
        one = (np.random.default_rng(1).random(1024) + 0j).astype(np.complex64)
        for _ in range(20):
            plans[10].process(one)
        t0 = time.perf_counter()
        for _ in range(200):
            plans[10].process(one)
        lat_us = (time.perf_counter() - t0) / 200 * 1e6
        per_dir = step_bytes / 2 / e2e_s / 1e9
        e2e = {"value": round(step_flops * world / e2e_s / 1e9, 1), "unit": "GFLOP/s",
               "h2d_bytes_per_step": int(step_bytes // 2) * world, "d2h_bytes_per_step": int(step_bytes // 2) * world,
               "ms_per_step": round(e2e_s * 1e3, 1), "steps": args.e2e_steps,
               "gbs_per_direction": round(per_dir, 1), "link_gbs_per_direction_concurrent": round(link, 1),
               "frac_of_link": round(per_dir / link, 3),
               "pageable": {"value": round(step_flops * world / pg_s / 1e9, 1), "unit": "GFLOP/s", "ms_per_step": round(pg_s * 1e3, 1),
                            "gbs_per_direction": round(step_bytes / 2 / pg_s / 1e9, 1)},
               "process_latency_us_n1024_batch1": round(lat_us, 1), "numa_binding": numa,
               "how": "b200fft_exec_host_outofplace on pinned host buffers (wall clock incl. H2D+D2H), "
                      f"{args.e2e_pinned_gib} GiB window reused per call; `pageable`: the same from numpy-allocated memory"}

    # ---- the other BASELINE configs, device resident, informational (not part of `value`) --------------
    extras = None
    if not args.no_extras:
        extras = []

        def timed(fn, reps):
            fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps

        # config 3: f64 forward + inverse round trip, N = 1234, batch = 1024 (in place)
        p64 = rb.FftPlanner(np.complex128, device=local_rank)
        f3, i3 = p64.plan_fft_forward(1234), p64.plan_fft_inverse(1234)
        x3 = torch.view_as_complex(torch.rand(64 * 1024 * 1234, 2, device=dev, dtype=torch.float64)).contiguous()

        def c3():
            for k in range(64):  # 64 distinct 19 MiB batches (1.2 GiB): no L2 reuse between calls
                sl = x3[k * 1024 * 1234:(k + 1) * 1024 * 1234]
                f3.process_device(sl)
                i3.process_device(sl)

        ms = timed(c3, 2) / 64
        extras.append({"config": "f64 forward+inverse N=1234 batch=1024", "plan": f3.describe(), "ms": round(ms, 4),
                       "gflops": round(2 * 5 * 1234 * math.log2(1234) * 1024 / (ms * 1e-3) / 1e9, 1),
                       "frac": round(2 * 32.0 * 1234 * 1024 / (ms * 1e-3) / 1e9 / hbm, 4)})
        del x3
        # config 4: f32 prime N = 65537, batch = 512
        f4 = planner.plan_fft_forward(65537)
        x4 = src[: 8 * 512 * 65537]
        y4 = dst[: 8 * 512 * 65537]

        def c4():
            for k in range(8):  # 8 distinct 256 MiB batches
                f4.process_device(x4[k * 512 * 65537:(k + 1) * 512 * 65537], out=y4[k * 512 * 65537:(k + 1) * 512 * 65537])

        ms = timed(c4, 2) / 8
        extras.append({"config": "f32 prime N=65537 batch=512", "plan": f4.describe(), "ms": round(ms, 4),
                       "gflops": round(5 * 65537 * math.log2(65537) * 512 / (ms * 1e-3) / 1e9, 1),
                       "frac": round(16.0 * 65537 * 512 / (ms * 1e-3) / 1e9 / hbm, 4)})
        # config 5: f32 N = 2^16, batch = 65536 sharded over the ranks of this job (65536 / world per GPU)
        per_rank = 65536 // world
        f5 = plans[16]
        ws5 = torch.empty(max(f5.workspace_bytes(per_rank), 16), dtype=torch.uint8, device=dev)

        def c5():
            f5.process_device(src[: per_rank << 16], out=dst[: per_rank << 16], workspace=ws5)

        barrier()
        ms = timed(c5, 2)
        if dist:
            tt = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = tt.item()
        extras.append({"config": f"f32 N=2^16 batch=65536 sharded over {world} GPU(s) ({per_rank} per GPU, shards resident)",
                       "plan": f5.describe(), "ms": round(ms, 4),
                       "gflops": round(5 * 65536 * 16 * 65536 / (ms * 1e-3) / 1e9, 1),
                       "frac_per_gpu": round(16.0 * 65536 * per_rank / (ms * 1e-3) / 1e9 / hbm, 4)})

        # f64 forward sweep (the same device path; 2^14 and up are two-pass plans of chunked launch pairs in f64)
        try:
            src64 = src.view(torch.float32).view(torch.complex128)
            dst64 = dst.view(torch.float32).view(torch.complex128)
            rows64, tot_b, tot_ms = [], 0.0, 0.0
            for lg in range(10, 19):
                n = 1 << lg
                f = p64.plan_fft_forward(n)
                ws64 = torch.empty(max(f.workspace_bytes(BATCH), 16), dtype=torch.uint8, device=dev)
                off = ((lg - 10) * (1 << 27)) % max(1, src64.numel() - BATCH * n)  # a different region per size

                def c64():
                    f.process_device(src64[off: off + BATCH * n], out=dst64[off: off + BATCH * n], workspace=ws64)

                ms = timed(c64, 3)
                rows64.append({"log2n": lg, "plan": f.describe(), "ms": round(ms, 4), "frac": round(32.0 * n * BATCH / (ms * 1e-3) / 1e9 / hbm, 4)})
                tot_b += 32.0 * n * BATCH
                tot_ms += ms
                del ws64
            extras.append({"config": "f64 forward N=2^10..2^18 batch=4096 (informational)", "ms": round(tot_ms, 3),
                           "frac": round(tot_b / (tot_ms * 1e-3) / 1e9 / hbm, 4), "per_size": rows64})
        except Exception as e:  # pragma: no cover
            extras.append({"config": "f64 sweep (informational)", "error": f"{type(e).__name__}: {e}"[:200]})

        # stated tolerance, as numbers: error of this library's output on the reference's test distribution (U[0,10), tests/accuracy.rs:86)
        # against an f64 numpy truth, per BASELINE config -- relative L2, and the largest element error in units of eps x the largest
        # output ("ulp of max"); `bound_rel_l2` is what the parity tests enforce (4 eps log2 N, tests/util.py)
        if rank == 0:
            try:
                acc = []

                def acc_row(name, pl, n, nb, dt, roundtrip=False):
                    rng = np.random.default_rng(n)
                    x = ((rng.random(n * nb) + 1j * rng.random(n * nb)) * 10).astype(dt)
                    d = torch.from_numpy(x).to(dev)
                    f = pl.plan_fft_forward(n)
                    f.process_device(d)
                    eps = 5.96e-8 if dt == np.complex64 else 1.11e-16
                    if roundtrip:
                        pl.plan_fft_inverse(n).process_device(d)
                        got = d.cpu().numpy().astype(np.complex128) / n
                        ref = x.astype(np.complex128)
                    else:
                        got = d.cpu().numpy().astype(np.complex128)
                        ref = np.fft.fft(x.astype(np.complex128).reshape(nb, n), axis=1).ravel()
                    err = (got - ref).reshape(nb, n)
                    refm = ref.reshape(nb, n)
                    # largest element error in units of eps x the largest output magnitude (the L-infinity form of the usual FFT error
                    # bound: every butterfly rounds relative to partial sums as large as the DC bin, N x mean of a U[0,10) signal), and the
                    # DC bin's own relative error
                    big = float(np.max(np.abs(refm)))
                    row = {"config": name, "plan": f.describe(), "rel_l2": float(f"{np.linalg.norm(err) / np.linalg.norm(refm):.3e}"),
                           "max_err_ulp_of_max": round(float(np.max(np.abs(err))) / (eps * big), 2),
                           "bound_rel_l2": float(f"{4 * eps * max(1.0, np.log2(n)) * (2 if roundtrip else 1):.3e}")}
                    if not roundtrip:
                        row["dc_bin_rel_err_ulp"] = round(float(np.max(np.abs(err[:, 0]) / np.abs(refm[:, 0]))) / eps, 2)
                    acc.append(row)

                for lg in (10, 15, 20):
                    acc_row(f"f32 forward N=2^{lg}", planner, 1 << lg, 4 if lg < 20 else 1, np.complex64)
                acc_row("f64 forward+inverse N=1234 (x/N vs input)", p64, 1234, 8, np.complex128, roundtrip=True)
                acc_row("f64 forward N=1234", p64, 1234, 8, np.complex128)
                acc_row("f32 prime N=65537", planner, 65537, 2, np.complex64)
                acc_row("f32 N=2^16", planner, 1 << 16, 4, np.complex64)
                extras.append({"config": "accuracy (stated tolerance as measured numbers)", "rows": acc})
            except Exception as e:  # pragma: no cover
                extras.append({"config": "accuracy", "error": f"{type(e).__name__}: {e}"[:200]})

        # config 5 as north_star states it (only with > 1 rank): the whole batch starts on GPU 0, NCCL point-to-point scatter of
        # contiguous batch shards over NVLink -> every rank transforms its shard -> gather back to GPU 0; the three stages
        # are timed separately (device events, max over ranks) and sampled transforms are checked against the CPU oracle
        if dist:
            try:
                from rustfft_b200.sharded import ShardedFft

                sh = ShardedFft(planner, 1 << 16)
                B5 = 65536
                full = src[: B5 << 16] if rank == 0 else None
                lo5, hi5 = sh.my_range(B5)

                def ev_ms(fn):
                    barrier()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    r = fn()
                    e1.record()
                    torch.cuda.synchronize()
                    tt = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                    return r, tt.item()

                stage_ms = {"scatter": [], "fft": [], "gather": []}
                for it in range(3):  # first pass = warm-up (NCCL channel setup), the other two are averaged
                    shard, t_s = ev_ms(lambda: sh.scatter(full, B5, root=0, device=dev, dtype=torch.complex64))
                    _, t_f = ev_ms(lambda: sh.process_local(shard))
                    _, t_g = ev_ms(lambda: sh.gather(shard, B5, root=0, out=dst if rank == 0 else None))
                    if it:
                        stage_ms["scatter"].append(t_s)
                        stage_ms["fft"].append(t_f)
                        stage_ms["gather"].append(t_g)
                    if it < 2:
                        del shard
                ms5 = {k: sum(v) / len(v) for k, v in stage_ms.items()}
                moved = (B5 - (hi5 - lo5 if rank == 0 else B5 // world)) * 65536 * 8.0  # bytes leaving / entering GPU 0
                row = {"config": f"f32 N=2^16 batch=65536: NCCL scatter from GPU 0 -> FFT on {world} GPUs -> gather to GPU 0",
                       "plan": sh.fft.describe(), "ms_scatter": round(ms5["scatter"], 3), "ms_fft": round(ms5["fft"], 3),
                       "ms_gather": round(ms5["gather"], 3),
                       "root_egress_gbs": round(moved / (ms5["scatter"] * 1e-3) / 1e9, 1),
                       "root_ingress_gbs": round(moved / (ms5["gather"] * 1e-3) / 1e9, 1),
                       "gflops_fft_only": round(5 * 65536 * 16 * B5 / (ms5["fft"] * 1e-3) / 1e9, 1),
                       "gflops_with_scatter_gather": round(5 * 65536 * 16 * B5 / ((ms5["scatter"] + ms5["fft"] + ms5["gather"]) * 1e-3) / 1e9, 1),
                       "limiter": "GPU 0's NVLink egress (scatter) and ingress (gather): (world-1)/world of 32 GiB each way through one GPU's links"}
                if rank == 0:
                    import oracle

                    oracle.build()
                    worst = 0.0
                    for b in (0, B5 // world, B5 // 2 + 3, B5 - 1):  # first shard, first transform of rank 1's, a middle one, the last
                        xb = src[b << 16:(b + 1) << 16].cpu().numpy()
                        yb = dst[b << 16:(b + 1) << 16].cpu().numpy()
                        want = oracle.fft(xb, 1 << 16)
                        worst = max(worst, float(np.linalg.norm(yb - want) / np.linalg.norm(want)))
                    row["checked_vs_oracle"] = {"transforms": 4, "max_rel_l2": float(f"{worst:.3e}"), "bound": 4 * 5.96e-8 * 16,
                                                "ok": bool(worst <= 2 * 4 * 5.96e-8 * 16)}
                extras.append(row)
                del shard
            except Exception as e:  # pragma: no cover
                extras.append({"config": "config 5 with NCCL scatter/gather", "error": f"{type(e).__name__}: {e}"[:300]})

        # informational: composite lengths of small primes through the two-pass SmoothFourStep plans (not a BASELINE
        # config; guarded so that a problem here can never cost the bench line)
        try:
            for n6, b6 in ((44100, 16384), (1000000, 512)):
                f6 = planner.plan_fft_forward(n6)
                ws6 = torch.empty(max(f6.workspace_bytes(b6), 16), dtype=torch.uint8, device=dev)

                def c6():
                    f6.process_device(src[: b6 * n6], out=dst[: b6 * n6], workspace=ws6)

                ms = timed(c6, 3)
                extras.append({"config": f"f32 composite N={n6} batch={b6} (informational)", "plan": f6.describe(), "ms": round(ms, 4),
                               "gflops": round(5 * n6 * math.log2(n6) * b6 / (ms * 1e-3) / 1e9, 1),
                               "frac": round(16.0 * n6 * b6 / (ms * 1e-3) / 1e9 / hbm, 4)})
                del ws6
        except Exception as e:  # pragma: no cover
            extras.append({"config": "f32 composite lengths (informational)", "error": f"{type(e).__name__}: {e}"[:200]})

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        import oracle

        oracle.build()
        cores = host_threads()
        gcpu, tcpu, per_cpu = cpu_sample(cores, min_reps=5, target_s=0.2, logs=logs)
        cpu = {"value": round(gcpu, 2), "unit": "GFLOP/s", "cores": cores, "kind": "port",
               "sample": f"every N in 2^10..2^20 with batch = {per_cpu[0]['batch']} (the same workload), in place; passes shorter than 0.2 s timed >= 5 times "
                         f"(median), longer ones once ({tcpu:.1f} s of timed CPU work); C++ port of RustFFT's scalar planner path, {cores} pinned workers "
                         "(= usable CPUs: affinity capped by the cgroup quota), one batch slice each",
               "per_size": per_cpu}

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": round(value, 1), "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": round(step_ms, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "BASELINE configs[1]: f32 forward, N=2^10..2^20, batch=4096 per GPU, out of place, "
                                   "device resident", "sizes_log2": logs, "batch_per_gpu": BATCH,
                       "launch": launch_mode,
                       "l2_policy": "inputs larger than L2: each size has its own region of a 32 GiB buffer, "
                                    ">= 32 GiB of other traffic between two touches of any byte",
                       "per_size": per_size},
            "roofline": {"bound": "hbm", "achieved": round(achieved, 1), "peak": hbm, "unit": "GB/s",
                         "frac": round(achieved / hbm, 4), "traffic": traffic, "peak_source": peak_src,
                         "kernel": "whole step (every launch in it is one of this repo's FFT passes)",
                         "algorithmic_bytes_per_step": int(step_bytes), "dominant_kernel": dominant,
                         "traffic_note": "DRAM bytes of one step from the committed ncu launch list (dram__bytes_read+write, "
                                         "--cache-control none): mean bytes per CTA of every kernel x the CTAs of a step; "
                                         "profiles/traffic.json" if traffic else None},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks, "other_configs": extras,
        }), flush=True)
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--logs", default="", help="comma list of log2 sizes (debug); default 10..20")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the informational timings of BASELINE configs 3-5")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--e2e-pinned-gib", type=float, default=4.0)
    ap.add_argument("--no-graph", action="store_true", help="plain stream launches instead of CUDA-graph replay")
    ap.add_argument("--profile", action="store_true", help="short run for ncu: 1 warm-up, no e2e / cpu legs")
    ap.add_argument("--profile-cold", action="store_true", help="with --profile: no warm-up sweep at all (launch lists)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/fft_f32_forward_log2n<L>.npy: float32 (rows, 2^L, 2), "
                         "the same seeded choice of whole transforms (rows) of every size in every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.profile_cold:
        args.profile = True
    if args.profile or args.logs:
        args.no_extras = True
    if args.profile:
        args.no_e2e = args.no_cpu = True
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
