#!/usr/bin/env python
"""bench.py — fn evals/sec of compiled `pytensor.function(..., mode="CUDA")` graphs on B200, with parity, roofline and the
reference C linker beside every number.

Contract (DESIGN.md §7):
  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--skip a,b,...] [--dump-outputs DIR]

  N = 1 (plain `python bench.py`): headline = BASELINE.json configs[1] (cfg2, the 32-scalar-op fused Elemwise+CAReduce graph
      over fp32 (4096,4096)); a "step" is one evaluation of the compiled function.
        value     evals/s, inputs resident in HBM, device outputs: exactly K timed steps, issued as one uninterrupted
                  stream and split into min(--reps, K // 10) (at least one) consecutive windows by CUDA events; MEDIAN
                  over the windows of ms/step.  The steps alternate two input sets; the last one always runs on the first set (seed 1).
        e2e       evals/s through `pytensor.function(..., mode="CUDA")` with pinned HOST inputs and NumPy outputs
        roofline  achieved HBM GB/s of the dominant kernel over MEASURED_PEAKS.json
        parity    CUDA outputs vs the reference C linker's outputs on the SAME 4096^2 arrays
      and, always on: `metric_graph` (the 265-node Elemwise+Gemm+Scan graph BASELINE.json's metric names, n=64 and
      n=4096, with the C linker beside it), `cfg3` (MLP 4096^3: tcgen05 bf16 and the fp32-accurate default mode),
      `cfg4` (Scan T=1000), `sharded_logp` (cfg5 on one GPU) — each with parity at the benchmarked shape.  These, `e2e`
      and the per-node profile behind `roofline` time fixed step counts of their own: --steps sets the headline only.
  N > 1 (torchrun): headline = BASELINE.json configs[4] (cfg5): hierarchical logp+grad over world x 2^17 independent
      chains sharded along the batch axis, ONE all-reduce of the packed [logp, grads] (75 floats) per evaluation, issued
      from inside the captured CUDA graph.  value = world x evaluations/s of the per-GPU shard (weak scaling); the line
      also carries the 1-GPU base measured in the same run, a strong-scaling point (2^20 chains in total), parity of
      the collective against a host sum of the per-rank partials and of rank 0's partial against the C linker, the
      N-rank collective self-test, and cfg2 replicas under `others`.  Here the headline is --reps windows of K steps each,
      with a barrier before every window so that the slowest rank bounds each one.
  --impl reference: the reference's own C linker (mode="CVM") on the host cores, same config strings (rank 0 only).
  --dump-outputs DIR (N = 1): after the timed steps, the headline's outputs of the last timed step as DIR/e.npy and
      DIR/r.npy (see dump_outputs), so that two builds can be compared output for output.  --impl reference dumps its
      last step too, on the same first input set.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)
# a run writes nothing into the source tree, not even __pycache__/ for the modules that build() never imported
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

B_LOCAL = 1 << 17      # chains per GPU of the sharded logp+grad graph (2^20 at 8 GPUs)
PAR_ROWS = 512         # rows of the n=4096 metric graph the C linker evaluates for parity (rows are independent)
N_ROWS, N_GROUPS, N_COV = 1024, 64, 8
MIN_WINDOW_STEPS = 10  # each event recorded between two steps costs device time: keep it under ~1/10 of a window
DUMP_BYTES = 64 * 10**6  # --dump-outputs writes at most this much in all


def dump_outputs(dirname, named):
    """Write each output as `dirname/<name>.npy`, in float64 if it was computed in float64 and float32 otherwise.  Each
    output gets an equal share of DUMP_BYTES; a larger one is written as its elements at a fixed, seeded set of flat
    indices (sorted), the same in every run, so that dumps of the same arguments compare element for element."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in named.items():
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        keep = (DUMP_BYTES // len(named) - 1024) // a.itemsize  # 1 KiB of each share is left for the .npy header
        if a.size > keep:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


def _peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "bf16_tflops": d.get("bf16_tflops", 1590.0),
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def _ncu_traffic(kernel_prefix, pattern=("*prof_k3_final*_ncu_summary.csv", "*prof_ew*_ncu_summary.csv")):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
    capture summary of the same command (profiles/; the newest round's capture first); None when no capture is committed."""
    import csv
    import glob

    patterns = (pattern,) if isinstance(pattern, str) else tuple(pattern)
    paths = [p for pat in patterns for p in sorted(glob.glob(os.path.join(REPO, "profiles", pat)), reverse=True)]
    for path in paths:
        try:
            rows = list(csv.reader(open(path)))
            hdr, units = rows[0], rows[1]
            kn, rd, wr = hdr.index("Kernel Name"), hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            vals = [float(r[rd]) * scale.get(units[rd], 1.0) + float(r[wr]) * scale.get(units[wr], 1.0)
                    for r in rows[2:] if r[kn].startswith(kernel_prefix) and not r[kn].endswith("_fin")]
            if vals:
                return sum(vals) / len(vals)
        except Exception:  # noqa: BLE001
            continue
    return None


def workload_config(world):
    """`config` of the JSON line — built by ONE function so that both arms print the same object."""
    if world == 1:
        return {"workload": "cfg2 (BASELINE.json configs[1]): 32-scalar-op fused Elemwise+CAReduce graph, fp32 "
                            "(4096,4096) -> e (4096,4096) f32, r=e.sum(1) f32 (acc f64)",
                "l2": "two alternating input sets, 384 MiB working set > 126 MB L2",
                "parallelism": "1 GPU"}
    return {"workload": "cfg5 (BASELINE.json configs[4]): hierarchical-normal logp+grad, n=1024 data rows, J=64 groups, "
                        f"K=8 covariates, batch = {world} x 2^17 independent chains (fp32), outputs summed over the batch",
            "l2": "per-GPU parameter arrays 38.8 MB, two alternating input sets; shared data 45 KB",
            "parallelism": f"batch-sharded over {world} GPUs (2^17 chains per GPU, weak), one 75-float all-reduce per evaluation"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self.first_done = threading.Event()  # set when the first nvidia-smi call has returned (or failed)
        self._t = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self.first_done.set()
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._loop, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = max(float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[3 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons,
                "samples": len(self.samples)}


def pinned_like(arr):
    """NumPy array backed by page-locked host memory (cudaHostAlloc through the C-ABI)."""
    import ctypes

    from pytensor_b200.runtime import lib as L

    p = ctypes.c_void_p()
    L.check(L.lib().ptk_host_alloc_pinned(ctypes.byref(p), max(arr.nbytes, 1)), "pinned alloc")
    buf = (ctypes.c_char * arr.nbytes).from_address(p.value)
    out = np.frombuffer(buf, dtype=arr.dtype).reshape(arr.shape)
    out[...] = arr
    return out


def bind_to_gpu_numa_node(local_rank):
    """Pin this process (and therefore its page-locked staging buffers, first-touch) to the CPU cores of the NUMA node
    the GPU hangs off — PCIe copies from the far socket cost ~40 % of the bandwidth (VERDICT r1: e2e efficiency 0.57 at
    N=4 with every rank on node 0).  Returns a short description for the JSON line."""
    try:
        import torch

        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        dev_id = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev_id:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return {"numa_node": None}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = set(os.sched_getaffinity(0)) & set(cpus)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as e:  # noqa: BLE001
        return {"numa_node": None, "error": repr(e)[:80]}


# ---- parity helpers ---------------------------------------------------------------------------------------------------
def parity(got, exp, rtol=1e-5, atol=1e-5, note=None):
    """Closeness in the reference's own sense (`values_eq_approx`, pytensor/tensor/math.py:92-139): |g-e| <= atol+rtol|e|.
    Also reports max|g-e| relative to the output's scale (max|e|)."""
    worst_tol, worst_scale, ok = 0.0, 0.0, True
    for g, e in zip(got, exp):
        g, e = np.asarray(g, dtype=np.float64), np.asarray(e, dtype=np.float64)
        if g.shape != e.shape:
            return {"ok": False, "error": f"shape {g.shape} vs {e.shape}"}
        if e.size == 0:
            continue
        d = np.abs(g - e)
        worst_tol = max(worst_tol, float(np.max(d / (atol + rtol * np.abs(e)))))
        worst_scale = max(worst_scale, float(np.max(d) / max(float(np.max(np.abs(e))), 1e-30)))
        ok = ok and bool(np.all(np.isfinite(g) == np.isfinite(e)))
    out = {"ok": bool(ok and worst_tol <= 1.0), "max_err_over_tol": worst_tol, "max_rel_to_scale": worst_scale,
           "rtol": rtol, "atol": atol, "against": "reference C linker (mode=CVM), same arrays"}
    if note:
        out["note"] = note
    return out


def timed_windows(fn, steps, reps, sync, barrier=None):
    """`reps` windows of `steps` calls each, CUDA events on the VM stream; returns per-window ms/step."""
    import torch

    out = []
    for _ in range(reps):
        if barrier is not None:
            barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        sync()
        out.append(e0.elapsed_time(e1) / steps)
    return out


def timed_steps(fn, steps, windows, sync):
    """`steps` calls `fn(0..steps-1)` issued back to back, split into `windows` (at most steps // MIN_WINDOW_STEPS, at
    least one) consecutive windows of near-equal size by CUDA events on the VM stream, one synchronise at the end: the
    device never waits for the host between windows.  Returns per-window ms/step."""
    import torch

    windows = max(1, min(windows, steps // MIN_WINDOW_STEPS))
    bounds = [steps * w // windows for w in range(windows + 1)]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(windows + 1)]
    ev[0].record()
    for w in range(windows):
        for i in range(bounds[w], bounds[w + 1]):
            fn(i)
        ev[w + 1].record()
    sync()
    return [ev[w].elapsed_time(ev[w + 1]) / (bounds[w + 1] - bounds[w]) for w in range(windows)]


def window_stats(ms):
    a = np.sort(np.asarray(ms, dtype=np.float64))
    return {"n": int(a.size), "median_ms": float(np.median(a)), "min_ms": float(a[0]), "max_ms": float(a[-1]),
            "p10_ms": float(a[int(0.1 * (a.size - 1))]), "p90_ms": float(a[int(round(0.9 * (a.size - 1)))])}


# ---- reference arm ------------------------------------------------------------------------------------------------------
def reference_arm(args, rank, world):
    """The reference's own CPU implementation of the path: mode="CVM" on the host cores (rank 0 only)."""
    if rank != 0:
        return
    from oracle import cvm
    from pytensor_b200 import workloads as W

    pytensor = cvm.configure("float32")
    env = cvm.describe()
    if world == 1:
        ins, outs, make_args, meta = W.cfg2_fused_elemwise(args.n)
        f = pytensor.function(ins, outs, mode="CVM", trust_input=True)
        a = make_args()
        scale, sample, cores = 1.0, f"{args.steps} full evaluations of the workload", 1
    else:
        # one step = a bounded sample: 2^13 of the shard's 2^17 chains (the graph is linear in the batch), scaled
        Bs = 1 << 13
        ins, outs, make_args, meta = W.cfg5_logp_grad(B=Bs, n=N_ROWS, J=N_GROUPS, K=N_COV, dtype="float32", packed=True)
        f = pytensor.function(ins, outs, mode="CVM", trust_input=True)
        a = make_args(seed=20, B_local=Bs)
        scale = Bs / B_LOCAL
        sample = (f"each step evaluates 2^13 of a shard's 2^17 chains (the graph is linear in the batch); value = steps x "
                  f"{scale} shard-evaluations / time; one host, all cores available to BLAS")
        cores = env["cores"]
    for _ in range(max(1, args.warmup)):
        f(*a)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = f(*a)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("e", "r"), out)))
    v = args.steps * scale / dt
    print(json.dumps({
        "impl": "reference", "metric": "fn evals/sec", "value": v, "unit": "evals/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps / scale, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(world),
        "cpu_baseline": {"value": v, "unit": "evals/s", "cores": cores, "kind": "reference", "sample": sample, "env": env},
        "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---- secondary configs (always on at N=1; each with parity at the benchmarked shape) ---------------------------------
def _time_dev(f, dev_args, torch, steps, warm, reps=5):
    for _ in range(warm):
        f(*dev_args)
    torch.cuda.synchronize()
    ms = timed_windows(lambda i: f(*dev_args), steps, reps, torch.cuda.synchronize)
    return float(np.median(ms)), window_stats(ms)


def bench_cfg3(pytensor, W, cuda_mode, dev, torch, peaks, cvm):
    """configs[2]: 3-layer MLP 4096^3. bf16 tcgen05 mode and the default (fp32-accurate) mode, parity vs the C linker."""
    out = {}
    ins, outs, make_args, meta = W.cfg3_mlp(4096)
    host = make_args()
    a = [dev.to_device(x) for x in host]
    f_ref = pytensor.function(ins, outs, mode="CVM", trust_input=True)
    t0 = time.perf_counter()
    exp = f_ref(*host)
    f_ref(*host)
    cpu_s = (time.perf_counter() - t0) / 2
    for key, kw, steps, tol in (("bf16_tcgen05", {"gemm_precision": "bf16"}, 10, (2e-2, 2e-2)),
                                ("default_fp32", {}, 3, (1e-5, 1e-5))):
        f = pytensor.function(ins, outs, mode=cuda_mode(device_outputs=True, borrow_outputs=True, **kw), trust_input=True)
        ms, st = _time_dev(f, a, torch, steps, 4)
        got = [dev.to_host(f(*a)[0])]
        tf = meta["flops"] / (ms * 1e-3) / 1e12
        kern = sorted({type(s.impl).__name__ + ":" + str(getattr(s.impl, "precision", "")) for s in f.vm.executor.program.steps})
        out[key] = {"evals_per_s": 1e3 / ms, "ms": ms, "tflops": tf, "frac_of_bf16_peak": tf / peaks["bf16_tflops"],
                    "windows": st, "nodes": kern,
                    "parity": parity(got, exp, rtol=tol[0], atol=tol[1],
                                     note="bf16 operands, fp32 accumulate: tolerance 2e-2 on outputs in [-1,1]"
                                     if key.startswith("bf16") else None)}
        del f
    out["cpu_reference"] = {"evals_per_s": 1 / cpu_s, "cores": os.cpu_count(), "sample": "2 evaluations (sgemm chain, all cores)"}
    from pytensor_b200.vm import nodes_blas as _nb

    out["resident_weights"] = dict(_nb._stage_cache_stats, note="staged copies of unchanged weight tensors reused across calls")
    return out


def bench_cfg4(pytensor, W, cuda_mode, dev, torch, peaks, cvm):
    """configs[3]: Scan, 1000 steps, carried state (8192,512) fp32; parity at T=1000 on a (256,512) row slice of the SAME
    state (rows are independent, so the slice of the result is the result of the slice)."""
    out = {}
    ins, outs, make_args, meta = W.cfg4_scan(8192, 512, 1000)
    host = make_args()
    a = [dev.to_device(x) for x in host]
    f = pytensor.function(ins, outs, mode=cuda_mode(device_outputs=True, borrow_outputs=True), trust_input=True)
    ms, st = _time_dev(f, a, torch, 5, 3)
    got = dev.to_host(f(*a)[0])
    f_ref = pytensor.function(ins, outs, mode="CVM", trust_input=True)
    sl = [host[0][:256].copy()] + host[1:]
    t0 = time.perf_counter()
    exp = f_ref(*sl)[0]
    cpu_s = time.perf_counter() - t0
    out["persistent_final_state"] = {
        "evals_per_s": 1e3 / ms, "ms": ms, "windows": st,
        "state_bytes_per_step_over_time_GBs": 2 * meta["state_bytes"] * meta["n_steps"] / (ms * 1e-3) / 1e9,
        "hbm_algorithmic_GBs": meta["bytes"] / (ms * 1e-3) / 1e9,
        "parity": parity([got[:256]], [exp], note="T=1000, rows 0..255 of the (8192,512) state vs the C linker on that slice"),
        "cpu_reference": {"evals_per_s_full_state_extrapolated": 1 / (cpu_s * 32), "sample": "1 evaluation of a 256-row slice x32"}}
    del f
    ins, outs, make_args, meta = W.cfg4_scan(8192, 512, 1000, full_trace=True)
    f = pytensor.function(ins, outs, mode=cuda_mode(device_outputs=True, borrow_outputs=True), trust_input=True)
    ms, st = _time_dev(f, a, torch, 4, 3)
    out["full_trace"] = {"evals_per_s": 1e3 / ms, "ms": ms, "windows": st, "trace_bytes": meta["bytes"],
                         "hbm_write_GBs": meta["bytes"] / (ms * 1e-3) / 1e9,
                         "frac_of_hbm_peak": meta["bytes"] / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}
    del f, a
    torch.cuda.empty_cache()
    try:  # secondary: matmul recurrence h <- tanh(h @ W + b), W (512,512)
        ins, outs, make_args, meta = W.cfg4_scan(8192, 512, 1000, matmul=True)
        host = make_args()
        a = [dev.to_device(x) for x in host]
        f = pytensor.function(ins, outs, mode=cuda_mode(device_outputs=True, borrow_outputs=True), trust_input=True)
        ms, st = _time_dev(f, a, torch, 2, 2, reps=3)
        got = dev.to_host(f(*a)[0])
        f_ref = pytensor.function(ins, outs, mode="CVM", trust_input=True)
        exp = f_ref(host[0][:64].copy(), *host[1:])[0]
        out["matmul_recurrence"] = {"evals_per_s": 1e3 / ms, "ms": ms, "windows": st,
                                    "tflops": 2 * 8192 * 512 * 512 * 1000 / (ms * 1e-3) / 1e12,
                                    "node": sorted({type(s.impl).__name__ for s in f.vm.executor.program.steps}),
                                    "cuda_graph_replay": bool(f.vm.executor.last_from_graph),
                                    "parity": parity([got[:64]], [exp], rtol=1e-4, atol=1e-4,
                                                     note="T=1000 chained fp32 matmuls, rows 0..63 vs the C linker; "
                                                          "1e-4: rounding differences compound over 1000 steps")}
        del f
        f = pytensor.function(ins, outs, mode=cuda_mode(device_outputs=True, borrow_outputs=True, gemm_precision="bf16"),
                              trust_input=True)
        ms, st = _time_dev(f, a, torch, 2, 2, reps=3)
        got = dev.to_host(f(*a)[0])
        out["matmul_recurrence_bf16"] = {"evals_per_s": 1e3 / ms, "ms": ms, "windows": st,
                                         "tflops": 2 * 8192 * 512 * 512 * 1000 / (ms * 1e-3) / 1e12,
                                         "max_abs_diff_vs_reference_rows_0_63": float(np.abs(got[:64] - exp).max()),
                                         "cuda_graph_replay": bool(f.vm.executor.last_from_graph),
                                         "note": "opt-in CUDA_BF16 mode (bf16 operands, fp32 accumulate), no parity claim"}
        del f, a
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001
        out["matmul_recurrence"] = {"error": repr(e)[:300]}
    return out


def bench_metric_graph(pytensor, W, cuda_mode, dev, torch, peaks, cvm):
    """The graph BASELINE.json's `metric` names: 84 x tanh(h@W+b), a 16-step Scan, a Sum — 265 compiled nodes; n=64
    (overhead-bound) and n=4096 (throughput-bound), the reference C linker timed beside both."""
    out = {}
    cases = ((64, {}, 50, "n64"), (4096, {}, 2, "n4096"), (4096, {"gemm_precision": "bf16"}, 3, "n4096_bf16"))
    only = [c for c in os.environ.get("PTK_BENCH_METRIC_CASES", "").split(",") if c]   # developer runs: a subset of the cases
    for n, kw, steps, label in cases:
        if only and label not in only:
            continue
        ins, outs, make_args, meta = W.metric_graph(n=n)
        host = make_args()
        f = pytensor.function(ins, outs, mode=cuda_mode(device_outputs=True, borrow_outputs=True, **kw), trust_input=True)
        a = [dev.to_device(x) for x in host]
        ms, st = _time_dev(f, a, torch, steps, 3, reps=5 if n == 64 else 3)
        nn = len(f.maker.fgraph.toposort())
        rec = {"evals_per_s": 1e3 / ms, "ms": ms, "windows": st, "compiled_nodes": nn,
               "launches_per_eval_after_fusion": len(f.vm.executor.program.steps), "us_per_compiled_node": 1e3 * ms / nn,
               "cuda_graph_replay": bool(f.vm.executor.last_from_graph), "mode": kw.get("gemm_precision", "default (fp32-accurate)")}
        if n > 64:
            rec["tflops"] = 84 * 2 * n ** 3 / (ms * 1e-3) / 1e12
        if n == 64:
            a_p, host_p = a, host
        else:
            # parity input: rows 0..511 of the same x with the same weights.  Every row of h runs through the 84 layers and
            # the Scan independently of the others (only the final Sum mixes rows), so the C linker's work drops 8x — the
            # bench stays within a few minutes — while the CUDA kernels, tile shapes along N and K and per-row arithmetic
            # are those of the timed 4096-row evaluation.
            host_p = [np.ascontiguousarray(host[0][:PAR_ROWS])] + list(host[1:])
            a_p = [dev.to_device(host_p[0])] + list(a[1:])
        got = [dev.to_host(f(*a_p)[0])]
        if label != "n4096_bf16":
            f_ref = pytensor.function(ins, outs, mode="CVM", trust_input=True)
            if n == 64:
                exp = f_ref(*host_p)
                evs, k = cvm.time_function(f_ref, host_p, min_seconds=2.0, min_calls=5, max_calls=2000)
                rec["cpu_reference"] = {"evals_per_s": evs, "sample": f"{k} evaluations", "cores": os.cpu_count()}
            else:
                t0 = time.perf_counter()
                exp = f_ref(*host_p)
                dt = time.perf_counter() - t0
                rec["cpu_reference"] = {"evals_per_s": PAR_ROWS / n / dt, "cores": os.cpu_count(),
                                        "sample": f"1 evaluation of rows 0..{PAR_ROWS - 1} (84 sgemm {PAR_ROWS}x{n}x{n} on all cores), "
                                                  f"scaled by {PAR_ROWS}/{n} to the full graph"}
            out["_exp_" + str(n)] = exp
            scale_e = float(np.abs(np.asarray(exp[0])).max())
            rec["parity"] = parity(got, exp, rtol=1e-4, atol=1e-4 * max(scale_e, 1.0),
                                   note="84 chained fp32 GEMM layers summed over the rows: 1e-4 of the output scale (per-layer "
                                        "rounding differences of two fp32 GEMMs compound; DESIGN.md §6)"
                                        + ("" if n == 64 else f"; compared on rows 0..{PAR_ROWS - 1} of the timed input"))
            if n > 64:
                # yardstick: the same graph in float64 on the same numbers (this backend's fp64 FMA kernels, themselves
                # held to 1e-5/1e-8 against the C linker's dgemm in tests/test_gpu_blas.py).  Two fp32 evaluations of an
                # 84-layer chain summed over the rows cannot agree better than each agrees with the exact result.
                import pytensor as _pt_mod

                fx = _pt_mod.config.floatX
                _pt_mod.config.floatX = "float64"
                try:
                    ins64, outs64, mk64, _ = W.metric_graph(n=n, dtype="float64")
                    f64 = pytensor.function(ins64, outs64, mode=cuda_mode(device_outputs=True, borrow_outputs=True),
                                            trust_input=True)
                    h64 = mk64()
                    a64 = [dev.to_device(np.ascontiguousarray(h64[0][:PAR_ROWS]))] + [dev.to_device(v) for v in h64[1:]]
                    truth = dev.to_host(f64(*a64)[0]).astype(np.float64)
                    del f64, a64, h64
                finally:
                    _pt_mod.config.floatX = fx
                torch.cuda.empty_cache()
                scale = float(np.abs(truth).max())
                e_ours = float(np.abs(np.asarray(got[0], dtype=np.float64) - truth).max() / scale)
                e_ref = float(np.abs(np.asarray(exp[0], dtype=np.float64) - truth).max() / scale)
                rec["parity"]["vs_float64_evaluation"] = {
                    "ours_max_err_over_scale": e_ours, "reference_max_err_over_scale": e_ref,
                    "note": "informational yardstick: distance of each fp32 evaluation from the float64 one (same row slice)"}
        else:
            rec["parity"] = parity(got, out["_exp_4096"], rtol=5e-2, atol=5e-2) if "_exp_4096" in out else {}
            rec["parity"]["ok"] = None
            rec["parity"]["note"] = ("informational, no parity claim: bf16 operands through 84 chained layers and a sum over "
                                     "the rows (the opt-in CUDA_BF16 mode; the default mode above carries the parity bar)")
        out[label] = rec
        del f, a
        torch.cuda.empty_cache()
    for k in [k for k in out if k.startswith("_exp_")]:
        del out[k]
    return out


# ---- cfg5: batch-sharded logp+grad --------------------------------------------------------------------------------------
def cfg5_io(W, B):
    ins, outs, _, _ = W.cfg5_logp_grad(B=B, n=N_ROWS, J=N_GROUPS, K=N_COV, dtype="float32", packed=True)
    return ins, outs


def build_cfg5(pytensor, W, cuda_mode, B):
    ins, outs, make_args, meta = W.cfg5_logp_grad(B=B, n=N_ROWS, J=N_GROUPS, K=N_COV, dtype="float32", packed=True)
    f = pytensor.function(ins, outs, mode=cuda_mode(device_outputs=True, borrow_outputs=True), trust_input=True)
    return f, make_args, meta, ins, outs


def time_sharded(sh, argsets, steps, reps, torch, dist, warm=6):
    for i in range(warm):
        res = sh(*argsets[i % len(argsets)], presharded=True)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    ms = timed_windows(lambda i: sh(*argsets[i % len(argsets)], presharded=True), steps, reps, torch.cuda.synchronize, barrier)
    if dist is not None:
        t = torch.tensor(ms, device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)  # per window: the slowest rank
        ms = [float(x) for x in t.tolist()]
    return ms, res


def sharded_logp(pytensor, W, cuda_mode, dev, torch, dist, world, rank, steps, reps, collective, B_local=B_LOCAL,
                 check=False, cvm=None):
    """BASELINE.json configs[4]: batch = world x B_local chains, sharded along the batch axis, ONE packed all-reduce."""
    from pytensor_b200.sharded import ShardedSum

    f, make_args, meta, ins, outs = build_cfg5(pytensor, W, cuda_mode, B_local * world)
    host_sets = [make_args(seed=20 + rank + 100 * s, B_local=B_local) for s in range(2)]
    local = [[dev.to_device(a) for a in hs] for hs in host_sets]
    sh = ShardedSum(f, batch_arg_idx=[0, 1, 2, 3], collective=collective if world > 1 else "none")
    ms, res = time_sharded(sh, local, steps, reps, torch, dist)
    med = float(np.median(ms))
    rec = {"evals_per_s": 1e3 / med, "ms_per_eval": med, "windows": window_stats(ms),
           "chains_per_s": B_local * world * 1e3 / med, "global_batch": B_local * world, "per_gpu_batch": B_local,
           "n_rows": N_ROWS, "allreduce_floats": 1 + meta["P"], "nodes": len(f.maker.fgraph.toposort()),
           "launches_per_eval": len(f.vm.executor.program.steps),
           "program": [repr(s.impl)[:80] for s in f.vm.executor.program.steps][:12],
           "graph_replay": bool(f.vm.executor.last_from_graph), "collective": sh.describe() if world > 1 else None}
    if check:
        # (a) the collective: all-reduced vector vs a host fp64 sum of every rank's LOCAL partial (no collective)
        got = dev.to_host(sh(*local[0], presharded=True)[0]).astype(np.float64)
        f_loc, _, _, _, _ = build_cfg5(pytensor, W, cuda_mode, B_local)
        part = dev.to_host(f_loc(*local[0])[0]).astype(np.float64)
        if world > 1:
            gathered = [None] * world
            dist.all_gather_object(gathered, part)
            summed = np.sum(np.stack(gathered), axis=0)
        else:
            summed = part
        rec["parity"] = {"collective": parity([got], [summed], rtol=1e-5, atol=1e-5)}
        rec["parity"]["collective"]["against"] = "host fp64 sum of the per-rank partials (no collective)"
        rec["logp_sum"] = float(got[0])
        # (b) the compute: rank 0's local partial vs the reference C linker on rank 0's shard (full 2^17 chains)
        if rank == 0 and cvm is not None:
            f_ref = pytensor.function(ins, outs, mode="CVM", trust_input=True)
            t0 = time.perf_counter()
            exp = np.asarray(f_ref(*host_sets[0])[0], dtype=np.float64)
            cpu_s = time.perf_counter() - t0
            scale = np.abs(exp).max()
            rec["parity"]["rank0_vs_reference"] = parity([part], [exp], rtol=1e-5, atol=1e-5 * scale,
                                                         note="sums of 2^17 x (1024|64|8|1) fp32 terms; atol = 1e-5 x the "
                                                              "largest component")
            rec["cpu_reference"] = {"shard_evals_per_s": 1 / cpu_s, "sample": "1 evaluation of one 2^17-chain shard incl. "
                                    "first-call overhead", "cores": os.cpu_count()}
        rec["parity"]["ok"] = all(v.get("ok", True) for v in rec["parity"].values() if isinstance(v, dict))
        del f_loc
    return rec, f, sh, local, host_sets


def collective_selftest(dev, torch, dist, world, rank):
    """tests/test_gpu_collective.py's first half on THIS run's ranks: the one-shot NVLink all-reduce vs NCCL vs the closed
    form, over both buffer parities and two sizes."""
    from pytensor_b200.sharded import PeerAllReduce

    ar = PeerAllReduce(nmax=1024, dtype="float32")
    worst = 0.0
    for it in range(6):
        n = 75 if it % 2 == 0 else 1024
        x = dev.to_device((np.arange(n, dtype="float32") + 1) * (rank + 1) * (it + 1))
        ref = x.clone()
        dist.all_reduce(ref)
        got = dev.to_host(ar(x)).astype(np.float64)
        exact = (np.arange(n) + 1.0) * (it + 1) * sum(r + 1 for r in range(world))
        worst = max(worst, float(np.max(np.abs(got - exact) / exact)), float(np.max(np.abs(got - dev.to_host(ref)) / exact)))
    t = torch.tensor([worst], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return {"ranks": world, "rounds": 6, "max_rel_vs_closed_form_and_nccl": float(t.item()), "ok": float(t.item()) < 1e-6}


def e2e_cfg5(f_host, host_sets, steps, reps, torch, dist):
    """Host parameter arrays in (pinned), NumPy [logp, grads] out, through the public call."""
    pin = [[pinned_like(a) for a in hs] for hs in host_sets]
    for i in range(4):
        res = f_host(*pin[i % 2])
    out = []
    for _ in range(reps):
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(steps):
            res = f_host(*pin[i % 2])
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) / steps)
    if dist is not None:
        t = torch.tensor(out, device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out = [float(x) for x in t.tolist()]
    h2d = int(sum(a.nbytes for a in host_sets[0]))
    d2h = int(sum(np.asarray(r).nbytes for r in res))
    return float(np.median(out)), h2d, d2h


# ---- cfg2 -----------------------------------------------------------------------------------------------------------------
def bench_cfg2(args, pytensor, W, cuda_mode, dev, jit, torch, dist, world, rank, local_rank, cvm, reps, want_cpu):
    ins, outs, make_args, meta = W.cfg2_fused_elemwise(args.n)
    f_dev = pytensor.function(ins, outs, mode=cuda_mode(device_outputs=True, borrow_outputs=True), trust_input=True)
    f_host = pytensor.function(ins, outs, mode="CUDA", trust_input=True)
    host_args = [make_args(1 + 10 * rank), make_args(101 + 10 * rank)]
    dev_args = [[dev.to_device(a) for a in s] for s in host_args]  # two input sets: 2 x 128 MiB > the 126 MB L2

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 6)  # eager+measure, capture, replay — for each of the two input sets
    for i in range(warm):
        f_dev(*dev_args[i % 2])
    barrier()
    ex = f_dev.vm.executor
    with ClockSampler(local_rank) as clocks:
        t_wait = time.perf_counter() + 3.0
        while not clocks.first_done.is_set() and time.perf_counter() < t_wait:
            for i in range(16):
                f_dev(*dev_args[i % 2])
            torch.cuda.synchronize()
        last = [None]

        def step(i):  # the two input sets alternate, and the last step runs on the first one
            last[0] = f_dev(*dev_args[(args.steps - 1 - i) % 2])

        barrier()
        ms_w = timed_steps(step, args.steps, reps, torch.cuda.synchronize)
        # the outputs are borrowed buffers that the next call overwrites: copy the last timed step's now
        dumped = dict(zip(("e", "r"), (dev.to_host(o) for o in last[0]))) if args.dump_outputs else None
        t_end = time.perf_counter() + 0.6
        while time.perf_counter() < t_end:  # keep the same load up so that later nvidia-smi samples see it
            for i in range(64):
                f_dev(*dev_args[i % 2])
            torch.cuda.synchronize()
    replayed = bool(ex.last_from_graph)
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    if dist is not None:
        t = torch.tensor(ms_w, device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_w = [float(x) for x in t.tolist()]
    ms = float(np.median(ms_w))
    value = world * 1e3 / ms

    # per-node device time: eager pass behind a queue filler so that host launch gaps do not pollute the events
    f_prof = pytensor.function(ins, outs, mode=cuda_mode(device_outputs=True, use_graph=False), trust_input=True)
    for i in range(3):
        f_prof(*dev_args[i % 2])
    torch.cuda.synchronize()
    exp_ = f_prof.vm.executor
    filler_src = dev.empty((1 << 28,), "float32")
    filler_dst = dev.empty((1 << 28,), "float32")
    for _ in range(6):
        dev.copy_strided(filler_dst, filler_src)
    l_before = jit.stats["launches"]
    exp_.event_log = []
    prof_steps = 12
    for i in range(prof_steps):
        f_prof(*dev_args[i % 2])
    torch.cuda.synchronize()
    launches_per_step = (jit.stats["launches"] - l_before) // prof_steps
    log, exp_.event_log = exp_.event_log, None
    del filler_src, filler_dst
    per_step = {}
    for i, a, b in log:
        per_step.setdefault(i, []).append(a.elapsed_time(b))
    step_ms = {i: float(np.median(v)) for i, v in per_step.items()}
    dom = max(step_ms, key=step_ms.get)
    dom_name = repr(exp_.program.steps[dom].impl)

    # e2e: host buffers through the public API
    pin_args = [[pinned_like(a) for a in s] for s in host_args]
    for i in range(max(4, args.warmup)):
        res = f_host(*pin_args[i % 2])
    e2e_steps = max(3, min(args.steps, 20))
    e2e_w = []
    for _ in range(5):
        barrier()
        t0 = time.perf_counter()
        for i in range(e2e_steps):
            res = f_host(*pin_args[i % 2])
        torch.cuda.synchronize()
        e2e_w.append((time.perf_counter() - t0) / e2e_steps)
    if dist is not None:
        t = torch.tensor(e2e_w, device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_w = [float(x) for x in t.tolist()]
    e2e_s = float(np.median(e2e_w))
    h2d = int(sum(a.nbytes for a in host_args[0]))
    d2h = int(sum(np.asarray(r).nbytes for r in res))

    peaks = _peaks()
    fused = "fused" in dom_name
    alg_bytes = meta["bytes"] if fused else 3 * 4 * args.n * args.n
    # duration of the dominant kernel: when a step IS one launch of it (the fused graph: a CUDA graph with that single
    # kernel node), its average duration over the timed region is the region's time per step — CUDA events around
    # K x reps launches, no per-launch event overhead; the per-launch event pair of the eager profile run (which
    # over-reads a ~40 us kernel by ~3 us) is reported beside it
    one_launch = launches_per_step == 1 and replayed
    kernel_ms = ms if one_launch else step_ms[dom]
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": _ncu_traffic("ptk_ew_red_row" if fused else "ptk_ew_vec"),
                "kernel": dom_name, "kernel_ms": kernel_ms, "algorithmic_bytes": alg_bytes, "peak_source": peaks["source"],
                "launches_per_step": launches_per_step,
                "how": ("one launch of this kernel per step: kernel_ms = CUDA-event time of the timed region / launches "
                        "(median over the windows)") if one_launch else
                       "median CUDA-event duration of the node's launch over 12 eager evaluations queued behind device work",
                "per_launch_event_pair": {"kernel_ms": step_ms[dom], "frac": alg_bytes / (step_ms[dom] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                                          "how": "median of an event pair around each launch, 12 eager evaluations queued "
                                                 "behind device work (includes the event overhead)"},
                "whole_graph": {"bytes": meta["bytes"], "gbs": meta["bytes"] / (ms * 1e-3) / 1e9,
                                "frac": meta["bytes"] / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "cuda_graph_replay": replayed}}

    cpu, par = None, None
    if want_cpu:
        f_ref = pytensor.function(ins, outs, mode="CVM", trust_input=True)
        exp = f_ref(*host_args[0])
        got_host = f_host(*pin_args[0])
        got_dev = [dev.to_host(o) for o in f_dev(*dev_args[0])]
        par = parity(got_dev, exp)
        par["host_path"] = parity(got_host, exp)["ok"]
        par["shape"] = f"({args.n},{args.n}) fp32: e and r=e.sum(1), the arrays the timed loop runs on"
        evs, n = cvm.time_function(f_ref, host_args[0], min_seconds=6.0, min_calls=3, max_calls=50)
        cpu = {"value": evs, "unit": "evals/s", "cores": 1, "kind": "reference",
               "sample": f"{n} full evaluations of the same workload (Elemwise/CAReduce C loops are single-threaded: "
                         "config.openmp=False)", "env": cvm.describe()}
    rec = {"value": value, "ms_per_step": ms, "windows": window_stats(ms_w),
           "e2e": {"value": world / e2e_s, "unit": "evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "steps": e2e_steps, "windows": 5,
                   "pipeline": ("chunked H2D|kernel|D2H x%d" % len(f_host.vm.executor._chunk_plan["bounds"]))
                   if f_host.vm.executor.chunked_calls else "one-shot"},
           "gpu_launches": launches_per_step * args.steps, "roofline": roofline, "cpu_baseline": cpu, "parity": par,
           "clocks": clocks.summary(),
           "timing": {"timed_steps": args.steps, "windows": len(ms_w),
                      "statistic": "median over windows of ms/step; the windows split one uninterrupted run of the "
                                   "timed steps (per window: max over ranks)"}}
    return rec


def bench_k1_stream(pytensor, cuda_mode, dev, torch, peaks):
    """Plain x + y over (4096,4096) fp32 through mode="CUDA": the streaming efficiency of the vector skeleton on its own."""
    import pytensor.tensor as pt

    x, y = pt.fmatrix("x"), pt.fmatrix("y")
    f = pytensor.function([x, y], x + y, mode=cuda_mode(device_outputs=True, borrow_outputs=True), trust_input=True)
    sets = [[dev.to_device(np.random.default_rng(s + k).standard_normal((4096, 4096)).astype("float32")) for k in range(2)]
            for s in (1, 11)]
    for i in range(6):
        f(*sets[i % 2])
    torch.cuda.synchronize()
    ms = timed_windows(lambda i: f(*sets[i % 2]), 20, 9, torch.cuda.synchronize)
    med = float(np.median(ms))
    gbs = 3 * 4096 * 4096 * 4 / (med * 1e-3) / 1e9
    return {"ms": med, "GBs": gbs, "frac_of_hbm_peak": gbs / peaks["hbm_gbs"], "windows": window_stats(ms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=25,
                    help="N = 1: windows the --steps timed steps are split into (at most --steps // 10); N > 1: "
                         "windows of --steps steps each (median reported)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip", default="", help="comma list of: metric,cfg3,cfg4,cfg5,k1,cfg2 (developer runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (one GPU only)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    skip = {s for s in args.skip.split(",") if s}
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        ap.error("--dump-outputs measures one GPU")

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch

    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else {"numa_node": None, "note": "single process: not bound"}
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from oracle import cvm  # configures PYTENSOR_FLAGS for the host framework (compile dir, BLAS); also the checker

    pytensor = cvm.configure("float32")
    import pytensor_b200  # noqa: F401
    from pytensor_b200 import workloads as W
    from pytensor_b200.link.cuda import cuda_mode
    from pytensor_b200.runtime import device as dev
    from pytensor_b200.runtime import jit

    dev.device()
    peaks = _peaks()
    reps = max(int(args.reps), 3)
    want_cpu = rank == 0 and world == 1 and not args.no_cpu_baseline

    def guarded(fn, *a, **k):
        try:
            return fn(*a, **k)
        except Exception as e:  # noqa: BLE001
            import traceback

            return {"error": repr(e)[:400], "where": traceback.format_exc().strip().splitlines()[-3:]}

    base = {"metric": "fn evals/sec", "unit": "evals/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world), "timing": {"windows": reps, "steps_per_window": args.steps,
                                                         "statistic": "median over windows (per window: max over ranks)"}}

    if world == 1:
        c2 = bench_cfg2(args, pytensor, W, cuda_mode, dev, jit, torch, dist, world, rank, local_rank, cvm, args.reps,
                        want_cpu)
        line = dict(base)
        for k in ("value", "ms_per_step", "windows", "e2e", "gpu_launches", "roofline", "cpu_baseline", "parity", "clocks",
                  "timing"):
            line[k] = c2[k]
        torch.cuda.empty_cache()
        if "k1" not in skip:
            line["k1_stream_add"] = guarded(bench_k1_stream, pytensor, cuda_mode, dev, torch, peaks)
        if "metric" not in skip:
            line["metric_graph"] = guarded(bench_metric_graph, pytensor, W, cuda_mode, dev, torch, peaks, cvm)
        if "cfg3" not in skip:
            line["cfg3"] = guarded(bench_cfg3, pytensor, W, cuda_mode, dev, torch, peaks, cvm)
        if "cfg4" not in skip:
            line["cfg4"] = guarded(bench_cfg4, pytensor, W, cuda_mode, dev, torch, peaks, cvm)
        if "cfg5" not in skip:
            def one_gpu_cfg5():
                rec, f, sh, local, host_sets = sharded_logp(pytensor, W, cuda_mode, dev, torch, None, 1, 0, 20, 9, "none",
                                                            check=True, cvm=cvm if want_cpu else None)
                f_host = pytensor.function(*cfg5_io(W, B_LOCAL), mode="CUDA", trust_input=True)
                s, h2d, d2h = e2e_cfg5(f_host, host_sets, 10, 5, torch, None)
                rec["e2e"] = {"value": 1 / s, "unit": "evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}
                return rec
            line["sharded_logp"] = guarded(one_gpu_cfg5)
        print(json.dumps(line))
        return

    # ---- N > 1: the batch-sharded logp+grad graph is the headline ------------------------------------------------------
    line = dict(base)
    line["numa"] = numa
    selftest = guarded(collective_selftest, dev, torch, dist, world, rank)
    # 1-GPU base of the weak-scaling series, measured in this very run: rank 0 alone, no collective, same per-GPU work
    base1 = None
    if rank == 0:
        r1, f1, _, _, _ = sharded_logp(pytensor, W, cuda_mode, dev, torch, None, 1, 0, args.steps, max(5, reps // 3), "none")
        base1 = {"value": r1["evals_per_s"], "ms_per_eval": r1["ms_per_eval"], "windows": r1["windows"],
                 "note": "rank 0 alone: one 2^17-chain shard, no collective (the N=1 point of the weak-scaling series)"}
        del f1
    dist.barrier()
    with ClockSampler(local_rank) as clocks:
        rec, f, sh, local, host_sets = sharded_logp(pytensor, W, cuda_mode, dev, torch, dist, world, rank, args.steps, reps,
                                                    "oneshot_ingraph", check=True, cvm=cvm)
    med = rec["ms_per_eval"]
    line.update({"value": world * 1e3 / med, "ms_per_step": med, "windows": rec["windows"], "clocks": clocks.summary(),
                 "parity": rec.pop("parity", None), "collective_selftest": selftest, "weak_scaling_base_1gpu": base1})
    launches = len(f.vm.executor.program.steps)
    line["gpu_launches"] = launches * args.steps * reps
    alg = sum(a.nbytes for a in host_sets[0]) + 4 * 75
    dom_ms = guarded(lambda: dominant_kernel_ms(f, local[0], dev, torch))
    if isinstance(dom_ms, tuple):
        line["roofline"] = {"bound": "hbm", "achieved": alg / (dom_ms[1] * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": alg / (dom_ms[1] * 1e-3) / 1e9 / peaks["hbm_gbs"], "traffic": _ncu_traffic("ptk_rowfuse", "*cfg5*_ncu_summary.csv"),
                            "kernel": dom_ms[0], "kernel_ms": dom_ms[1], "algorithmic_bytes": alg, "peak_source": peaks["source"],
                            "note": "the fused likelihood kernel reads every parameter once (B x 74 floats) and does ~46 flop "
                                    "per (chain, data row): it is fp32-issue-bound, not HBM-bound — see DESIGN.md §4"}
    line["sharded_logp"] = rec
    # alternatives: NCCL all-reduce after the replay, one-shot kernel after the replay
    alts = {}
    for coll in ("nccl", "oneshot"):
        r = guarded(lambda c=coll: sharded_logp(pytensor, W, cuda_mode, dev, torch, dist, world, rank, args.steps,
                                                 max(5, reps // 3), c)[0])
        alts[coll] = {k: r.get(k) for k in ("evals_per_s", "ms_per_eval", "windows", "collective", "error") if k in r}
    line["collective_alternatives"] = alts
    # strong scaling: 2^20 chains in total, 2^20 / world per GPU
    line["strong_scaling"] = guarded(lambda: {k: v for k, v in sharded_logp(
        pytensor, W, cuda_mode, dev, torch, dist, world, rank, args.steps, max(5, reps // 3), "oneshot_ingraph",
        B_local=(1 << 20) // world)[0].items() if k in ("evals_per_s", "ms_per_eval", "windows", "global_batch", "per_gpu_batch")})
    # e2e: host parameter arrays through the public call + the all-reduce
    def e2e_multi():
        from pytensor_b200.sharded import ShardedSum

        f_h = pytensor.function(*cfg5_io(W, B_LOCAL * world),
                                mode=cuda_mode(device_outputs=True, borrow_outputs=True), trust_input=True)
        shh = ShardedSum(f_h, [0, 1, 2, 3], collective="oneshot_ingraph")

        def call(*a):
            return [dev.to_host(shh(*a, presharded=True)[0])]
        s, h2d, d2h = e2e_cfg5(call, host_sets, 10, 5, torch, dist)
        return {"value": world / s, "unit": "evals/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "note": "per rank: pinned host parameter arrays -> device (inside the call), graph replay incl. the "
                        "all-reduce, 75 floats back to the host"}
    line["e2e"] = guarded(e2e_multi)
    # cfg2 replicas (the round-1 headline) as an extra
    if "cfg2" not in skip:
        c2 = guarded(bench_cfg2, args, pytensor, W, cuda_mode, dev, jit, torch, dist, world, rank, local_rank, cvm,
                     max(5, reps // 3), False)
        line["others"] = {"cfg2_replicas": {k: c2.get(k) for k in ("value", "ms_per_step", "windows", "e2e", "roofline", "error")
                                            if k in c2}}
    if rank == 0:
        print(json.dumps(line))
    dist.destroy_process_group()


def dominant_kernel_ms(f, dev_args, dev, torch):
    """(name, ms) of the longest step of one eager evaluation of `f` (CUDA events around each node)."""
    ex = f.vm.executor
    ug, ex.use_graph = ex.use_graph, False
    try:
        for _ in range(2):
            f(*dev_args)
        torch.cuda.synchronize()
        ex.event_log = []
        for _ in range(6):
            f(*dev_args)
        torch.cuda.synchronize()
        log, ex.event_log = ex.event_log, None
    finally:
        ex.use_graph = ug
    per = {}
    for i, a, b in log:
        per.setdefault(i, []).append(a.elapsed_time(b))
    med = {i: float(np.median(v)) for i, v in per.items()}
    dom = max(med, key=med.get)
    return repr(ex.program.steps[dom].impl)[:100], med[dom]


if __name__ == "__main__":
    main()
