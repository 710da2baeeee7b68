#!/usr/bin/env python
"""bench.py -- Opt fit (orthant NNLS enumeration) throughput on B200, one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--workload NAME]
                  [--no-cpu-baseline] [--no-extras] [--dump-outputs DIR]

BASELINE.json's metric is "Opt fit time-to-solution and orthant NNLS solves/sec at K=20, 1/2/4/8 B200":
every N runs the SAME problem -- `k20_m200`: synthetic N=100 000, M=200, K=20, eta=1e-3 -- so the series
over N is STRONG scaling (rows of X sharded for K1/K4, the sign-pattern range split N ways for K2, winners
gathered).

A "step" is one complete Opt fit: Gram build (K1) -> orthant NNLS solves (K2) -> argmin (K3) -> data-space
recompute of the winner (K4).  `value` = NNLS problems solved per second with the data set resident in HBM,
counting 2^K problems per fit (SURVEY.md 8d: the intercept sign is left FREE inside each solve, so one
problem per sign pattern of the K user groups resolves the two reference orthants that differ only in the
intercept sign; `reference_orthants_per_sec` = 2 x value is the rate in the reference's own 2^(K+1) count).
`e2e` = the same through pls_load + the fit with HOST (pinned) buffers: the host->device copy of X, y, P and
the device->host read of the result are inside the timed region.

Extras inside the same JSON line (`extra`): at N = 1 the configs[1] workload (cfg2: K=16, the config the
round-1 numbers were quoted on) and the end-to-end time from PAGEABLE host memory; at N > 1 the same K=20
fit driven by ONE process through the in-library multi-GPU path (pls_create with N devices, what a Julia
host uses), run by rank 0 after the timed region while the other ranks wait on a CPU barrier; at N = 8 also
BASELINE configs[2] in full (N=1M, M=512, K=24) on that path.

--impl reference: the reference's own CPU algorithm (oracle/pls_oracle.c: per-orthant materialised column
scaling + data-space Lawson-Hanson + residual norm, i.e. Opt.jl:85-94) on all host threads, on a bounded
sample of the same workload's orthants, in the same unit (it spends two of its NNLS solves per sign pattern).
Julia is not in this image, so this is the C restatement ("port"); it never loads the product library.

--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step returned as DIR/<name>.npy
(float64), so that two builds can be compared output for output on the same seeded inputs.  Native arm: the
fit's winner `b_best`, its objective `opt` and its raw weights `alpha_raw` (M+1).  Reference arm: the sampled
orthants `b_list` and their objectives `objs`.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

_JSON_OUT = sys.stdout
METRIC = "opt_fit_orthant_nnls_solves_per_sec"
UNIT = "nnls_problems/s"   # sign patterns of the K user groups resolved per second = 2^K per fit (both arms)
DEFAULT_WORKLOAD = "k20_m200"

K2_KERNELS = {
    1: "k2_orthant_chains (single-pivot active set, rank-1 updates of a dense inverse)",
    3: "k2v3_orthant_chains (one-level block principal pivoting, DMMA rank-8 updates of the packed inverse)",
    4: "k2v4_orthant_ranges (two-level: per-CTA swept tableau + block pivoting on the fast Gray groups, CTA per chain)",
    5: "k2v5_orthant_walks (two swept tableaus per Gray walk: T1 in L2/HBM changed only by rank-8 DMMA folds, a small tile-packed T2 in shared memory swept by DMMA block pivots; one small CTA per walk)",
}


def load_synth():
    """synth.py on its own -- the reference arm must not map the product library into its process."""
    spec = importlib.util.spec_from_file_location("pls_synth_standalone", os.path.join(entry.PKG_DIR, "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "source": "fallback"}
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            peaks.update(json.load(open(p)))
            peaks["source"] = "measured"
        except Exception:
            pass
    # FP64 peaks are not in MEASURED_PEAKS.json: measured by tools/fp64_peak.cu on this pool's B200
    p64 = os.path.join(ROOT, "profiles", "fp64_peaks_r01.json")
    peaks["fp64"] = json.load(open(p64)) if os.path.exists(p64) else {"dfma_tflops": 36.4, "dmma_m8n8k4_tflops": 37.1}
    return peaks


def ncu_dram_traffic(workload, variant, threads):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed
    `ncu --set full` capture -- used only if that capture was taken on THIS workload with THIS kernel variant
    and CTA size (profiles/k2_traffic.json lists the captures); otherwise None."""
    p = os.path.join(ROOT, "profiles", "k2_traffic.json")
    if not os.path.exists(p):
        return None, None
    try:
        for e in json.load(open(p)):
            if e["workload"] == workload and int(e["k2_variant"]) == int(variant) and int(e["k2_threads"]) == int(threads):
                return float(e["dram_bytes_per_launch"]), e.get("source")
    except Exception:
        pass
    return None, None


class ClockSampler:
    """Samples SM clocks and throttle reasons during the timed region (pynvml)."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40,
                 "sw_thermal_slowdown": 0x20, "hw_power_brake": 0x80, "sync_boost": 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        if self.nv:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        if self._thr:
            self._stop.set()
            self._thr.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def make_workload(name, synth):
    N, M, K, eta, seed, mixed = synth.CONFIGS[name]
    X, y, P = synth.make_synthetic(N, M, K, seed, mixed_sign=mixed)
    wl = {"workload": f"{name}: synthetic N={N} M={M} K={K} eta={eta} fit(Opt).  2^K={1 << K} NNLS problems per fit -- one per sign "
                      f"pattern of the K user groups, intercept sign free (SURVEY.md 8d); each resolves the two orthants of the "
                      f"reference's 2^(K+1)={1 << (K + 1)} enumeration that differ only in the intercept sign (same b*, alpha, "
                      f"objective: tests/test_gpu_parity.py::test_paired_orthants_*).  `value` counts the 2^K problems",
          "N": N, "M": M, "K": K, "eta": eta, "nnls_problems_per_fit": 1 << K, "reference_orthants_per_fit": 1 << (K + 1),
          "seed": seed,
          "l2": "inputs larger than L2 (Z = %.0f MB) and an L2 flush (256 MB memset) before every timed step" % (N * (M + 2) * 8 / 1e6)}
    return X, y, P, eta, wl


def cpu_reference_sample(oc, X, y, P, eta, n_orthants, nthreads, seed=0):
    """Times the C restatement of the reference loop on `n_orthants` seeded random orthants (of the reference's
    2^(K+1)) at full N, M.  Returns (orthant solves per second, seconds, {b_list, objs})."""
    rng = np.random.default_rng(seed)
    bl = rng.integers(0, 1 << (P.shape[1] + 1), size=n_orthants).astype(np.int64)
    t0 = time.perf_counter()
    r = oc.opt_fit(X, y, P, eta, b_list=bl, nthreads=nthreads, want_alpha=False)
    dt = time.perf_counter() - t0
    return n_orthants / dt, dt, {"b_list": bl, "objs": r["objs"]}


def dump_outputs(out_dir, arrays):
    """Writes every array of `arrays` as out_dir/<name>.npy in float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_reference(args, rank, world):
    if rank != 0:
        return
    _, oc = entry.load_oracle()           # the library build() made: the tree may be read-only, so no rebuild here
    synth = load_synth()
    X, y, P, eta, wl = make_workload(args.workload or DEFAULT_WORKLOAD, synth)
    cores = oc.num_threads()
    per_step = cores                      # one orthant per host thread per step (~5-10 s)
    for i in range(args.warmup):
        cpu_reference_sample(oc, X, y, P, eta, max(1, per_step // 4), cores, seed=100 + i)
    t_tot, n_tot = 0.0, 0
    for i in range(args.steps):
        _, dt, last = cpu_reference_sample(oc, X, y, P, eta, per_step, cores, seed=i)
        t_tot += dt
        n_tot += per_step
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    orth = n_tot / t_tot
    val = orth / 2.0                      # the reference spends two NNLS solves (intercept sign -, +) per sign pattern
    sample = (f"{per_step} seeded random orthants per step at full N, M (of the reference's {1 << (P.shape[1] + 1)}); C restatement of "
              f"Opt.jl:85-94 (Julia not installed); {orth:.4g} orthant solves/s = {val:.4g} sign patterns/s")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": wl,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "reference_orthants_per_sec": orth,
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_JSON_OUT, flush=True)


def run_native(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    pkg = entry.load_package()
    from importlib import import_module
    synth = import_module(entry.PKG_NAME + ".synth")
    distmod = import_module(entry.PKG_NAME + ".dist")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    cudart = torch.cuda.cudart()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    cpu_group = dist.new_group(backend="gloo") if world > 1 else None
    comm = distmod.TorchComm(device=dev) if world > 1 else None
    ctx = pkg.Context(local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, sample_clocks, collective=True):
        """Times `steps` calls of fn on the device: CUDA events recorded on torch's current stream right
        before and right after each call.  The library call is blocking (it synchronises its own stream
        before it returns), so the closing event is reached only after all of the step's kernels and
        copies have finished; barrier + synchronize bracket every step.  Returns the max over ranks."""
        bar = barrier if collective else torch.cuda.synchronize
        for _ in range(warmup):
            fn()
        # one sampler for the job (rank 0's GPU): NVML queries from every rank at once contend with the CUDA driver calls of the
        # timed steps (an 8-rank run lost > 1 ms per step to them)
        sampler = ClockSampler(local_rank) if (sample_clocks and rank == 0) else None
        per_step, host_step, last = [], [], None
        bar()
        if sampler:
            sampler.start()
        for _ in range(steps):
            flush.zero_()                  # L2 flush, outside the timed step
            bar()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            last = fn()
            e1.record()
            torch.cuda.synchronize()
            host_step.append(time.perf_counter() - t0)
            per_step.append(e0.elapsed_time(e1) * 1e-3)
        bar()
        clocks = sampler.stop() if sampler else None
        tt = torch.tensor([sum(per_step), sum(host_step)], dtype=torch.float64, device=dev)
        if world > 1 and collective:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        if clocks is not None:
            clocks["host_clock_s"] = float(tt[1].item())
        return float(tt[0].item()), last, clocks

    def measure(name, steps, warmup, sample_clocks, sharded):
        """resident + end-to-end timings of one workload on `ctx` (this rank's shard when sharded)."""
        X, y, P, eta, wl = make_workload(name, synth)
        N, M = X.shape
        K = P.shape[1]
        Mp = M + 1
        w_, r_ = (world, rank) if sharded else (1, 0)
        r0, r1 = (N * r_) // w_, (N * (r_ + 1)) // w_
        Xs = np.asfortranarray(X[r0:r1]); ys = np.ascontiguousarray(y[r0:r1]); Pc = np.asfortranarray(P)
        for a in (Xs, ys, Pc):
            cudart.cudaHostRegister(a.ctypes.data, a.nbytes, 0)

        def step_resident():
            if w_ == 1:
                r = ctx.opt_fit_resident()
                return r["b_best"], r["opt"], r["alpha_raw"], r["stats"]
            bb, obj, alpha = distmod.opt_fit_sharded(ctx, comm, Mp, K + 1)
            return bb, obj, alpha, ctx.stats()

        def step_e2e(Xh=Xs, yh=ys):
            if w_ == 1:
                r = ctx.opt_fit(Xh, yh, Pc, eta=eta, prepared=True)
                return r["b_best"], r["opt"], r["alpha_raw"], r["stats"]
            bb, obj, alpha = distmod.opt_fit_sharded(ctx, comm, Mp, K + 1,
                                                     reload=lambda: ctx.load(Xh, yh, Pc, eta=eta, prepared=True))
            return bb, obj, alpha, ctx.stats()

        ctx.load(Xs, ys, Pc, eta=eta, prepared=True)
        t_res, last, clocks = timed(step_resident, steps, warmup, sample_clocks, collective=sharded)
        t_e2e, last_e, _ = timed(step_e2e, steps, max(1, warmup // 2), False, collective=sharded)
        assert last_e[0] == last[0], "e2e and resident paths disagree on the winner"
        t_page = None
        if not sharded:                    # pageable host memory, as a Julia Array is: the driver stages the copy
            Xp = np.array(Xs, order="F", copy=True); yp = ys.copy()
            t_page, last_p, _ = timed(lambda: step_e2e(Xp, yp), steps, 1, False, collective=False)
            assert last_p[0] == last[0]
        for a in (Xs, ys, Pc):
            cudart.cudaHostUnregister(a.ctypes.data)
        h2d = int((Xs.nbytes + ys.nbytes + Pc.nbytes) * w_)
        return dict(X=X, y=y, P=P, eta=eta, wl=wl, t_res=t_res, t_e2e=t_e2e, t_page=t_page, last=last, clocks=clocks,
                    h2d=h2d, d2h=int((Mp + 4 + 10) * 8 * w_))

    name = args.workload or DEFAULT_WORKLOAD
    m = measure(name, args.steps, args.warmup, True, sharded=world > 1)
    X, y, P, eta, wl = m["X"], m["y"], m["P"], m["eta"], m["wl"]
    N, M = X.shape
    K = P.shape[1]
    bb, obj, alpha, st = m["last"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"b_best": bb, "opt": obj, "alpha_raw": alpha})
    extra = {}

    # ---- extras: never inside the timed region of the headline numbers ------------------------------------
    if not args.no_extras and world == 1:
        try:
            c2 = measure("cfg2", max(3, args.steps), 3, False, sharded=False)
            s2 = c2["last"][3]
            extra["cfg2"] = {
                "workload": c2["wl"]["workload"], "nnls_problems_per_fit": 1 << 16,
                "ms_per_step_resident": 1e3 * c2["t_res"] / max(3, args.steps), "ms_per_step_e2e_pinned": 1e3 * c2["t_e2e"] / max(3, args.steps),
                "ms_per_step_e2e_pageable": 1e3 * c2["t_page"] / max(3, args.steps),
                "nnls_problems_per_sec": (1 << 16) * max(3, args.steps) / c2["t_res"],
                "stages_ms": {"gram_k1": s2["ms_gram"], "nnls_k2_k3": s2["ms_nnls"], "recompute_k4": s2["ms_recompute"]},
                "k1_tflops": s2["gram_flops"] / (s2["ms_gram"] * 1e-3) / 1e12 if s2["ms_gram"] > 0 else None,
                "k2_variant": s2["k2_variant"], "result": {"b_best": int(c2["last"][0]), "opt": float(c2["last"][1])}}
        except Exception as e:      # an extra must never cost the headline line
            extra["cfg2"] = {"error": repr(e)}
    if not args.no_extras and world > 1:
        # the in-library multi-GPU path (one process, pls_create with `world` devices): rank 0 alone, the other
        # ranks wait on a CPU (gloo) barrier so that no NCCL kernel spins on their GPUs meanwhile
        if rank == 0:
            try:
                extra["single_process"] = single_process_fit(pkg, torch, list(range(world)), X, y, P, eta, args.steps, bb)
                if world == 8 and not os.environ.get("PLS_BENCH_SKIP_CFG3"):
                    extra["cfg3_single_process"] = cfg3_single_process(pkg, torch, synth, list(range(world)))
            except Exception as e:
                extra["single_process"] = {"error": repr(e)}
        dist.barrier(group=cpu_group)

    if rank != 0:
        return
    peaks = load_peaks()
    problems = 1 << K
    t_res, t_e2e = m["t_res"], m["t_e2e"]
    value = problems * args.steps / t_res
    e2e_val = problems * args.steps / t_e2e
    k2_ms = st["ms_nnls"]
    fp64_peak = float(peaks["fp64"].get("dfma_tflops", 36.4))
    k2_tflops = st["nnls_flops"] / (k2_ms * 1e-3) / 1e12 if k2_ms > 0 else 0.0
    traffic, traffic_src = ncu_dram_traffic(name, st["k2_variant"], st["k2_threads"])
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_res / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": wl,
        "clocks": m["clocks"],
        "e2e": {"value": e2e_val, "unit": UNIT, "ms_per_step": 1e3 * t_e2e / args.steps,
                "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"], "host_memory": "pinned (cudaHostRegister outside the timed region)"},
        "gpu_launches": int(st["kernel_launches"] * args.steps * world),
        "reference_orthants_per_sec": 2.0 * value,
        "roofline": {
            "kernel": K2_KERNELS.get(int(st["k2_variant"]), "k2 variant %d" % st["k2_variant"]) +
                      " <%d threads, %d CTAs/SM, grid %d>; FP64 DMMA/DFMA (tcgen05 has no f64 kind)" % (st["k2_threads"], st["k2_ctas_per_sm"], st["k2_grid"]),
            "k2_variant": int(st["k2_variant"]),
            "bound": "latency", "achieved": k2_tflops, "peak": fp64_peak, "unit": "TFLOP/s",
            "frac": k2_tflops / fp64_peak if fp64_peak else None, "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": "FP64 DFMA peak measured by tools/fp64_peak.cu on this pool (profiles/fp64_peaks_r01.json); MEASURED_PEAKS.json holds no FP64 figure",
            "algorithmic_flops_per_launch": st["nnls_flops"], "launch_ms": k2_ms,
            "flops_per_nnls_problem": st["nnls_flops"] / max(1, st["nnls_problems"]),
            "l2_model_gbs": st["nnls_l2_bytes"] / (k2_ms * 1e-3) / 1e9 if k2_ms > 0 else None,
            "note": "K2 is neither HBM- nor FLOP-bound: 16 B leave the chip per problem and the work is a chain of short dependent "
                    "steps on an L2-resident working set, so the binding limit is latency / issue rate (DESIGN.md 3).  achieved = the "
                    "kernel's own work counters (2 M' sum_p + 4 sum_p2) / launch time of rank 0's shard; frac is that against the "
                    "measured FP64 peak",
        },
        "stages_ms": {"gram_k1": st["ms_gram"], "nnls_k2_k3": st["ms_nnls"], "recompute_k4": st["ms_recompute"]},
        "k1_gram": {"tflops": st["gram_flops"] / (st["ms_gram"] * 1e-3) / 1e12 if st["ms_gram"] > 0 else None,
                    "peak_tflops": float(peaks["fp64"].get("dmma_m8n8k4_tflops", 37.1))},
        "solver_counters": {k: st[k] for k in ("pivots", "grad_evals", "sum_p", "sum_p2", "bpp_iters", "spills", "rebuilds", "blocked",
                                               "nnls_problems", "k2_max_drift")},
        "result": {"b_best": int(bb), "opt": float(obj)},
        "time_to_solution_ms": {"resident": 1e3 * t_res / args.steps, "from_pinned_host": 1e3 * t_e2e / args.steps,
                                "from_pageable_host": 1e3 * m["t_page"] / args.steps if m["t_page"] else None},
        "extra": extra,
    }
    if world == 1 and not args.no_cpu_baseline:
        _, oc = entry.load_oracle()
        n_s = 4
        v, dt, _ = cpu_reference_sample(oc, X, y, P, eta, n_s, 1, seed=0)
        line["cpu_baseline"] = {"value": v / 2.0, "unit": UNIT, "cores": 1, "kind": "port",
                                "sample": f"{n_s} seeded random orthants at full N, M, single thread (the reference loop is serial), {dt:.1f} s: "
                                          f"{v:.4g} orthant solves/s = {v / 2:.4g} sign patterns/s; C restatement of Opt.jl:85-94"}
    print(json.dumps(line), file=_JSON_OUT, flush=True)


def single_process_fit(pkg, torch, devices, X, y, P, eta, steps, b_expect):
    """The K=20 fit through pls_create(n_dev = len(devices)): one process, one host thread per device inside the
    library, Gram sums exchanged peer-to-peer.  Host-clock timings around the blocking call (all devices idle
    before and after)."""
    c = pkg.Context(devices)
    try:
        c.load(X, y, P, eta=eta)
        for _ in range(2):
            r = c.opt_fit_resident()
        ts = []
        for _ in range(max(3, steps)):
            for d in devices:
                torch.cuda.synchronize(d)
            t0 = time.perf_counter()
            r = c.opt_fit_resident()
            ts.append(time.perf_counter() - t0)
        st = r["stats"]
        K = P.shape[1]
        return {"devices": len(devices), "ms_per_step_resident": 1e3 * float(np.mean(ts)), "ms_best": 1e3 * float(np.min(ts)),
                "nnls_problems_per_sec": (1 << K) / float(np.mean(ts)), "same_winner_as_sharded_run": bool(r["b_best"] == b_expect),
                "stages_ms": {"gram_k1_and_exchange": st["ms_gram"], "nnls_k2_k3_max_over_devices": st["ms_nnls"], "recompute_k4": st["ms_recompute"]},
                "k2_variant": st["k2_variant"], "timing": "host clock around the blocking pls_opt_fit_resident call"}
    finally:
        c.close()


def cfg3_single_process(pkg, torch, synth, devices):
    """BASELINE configs[2] in full: N=1M, M=512, K=24, fit(Opt), 2^24 NNLS problems (2^25 reference orthants)."""
    N, M, K, eta, seed, mixed = synth.CONFIGS["cfg3"]
    t0 = time.perf_counter()
    X, y, P = synth.make_synthetic_parallel(N, M, K, seed)
    t_gen = time.perf_counter() - t0
    c = pkg.Context(devices)
    try:
        t0 = time.perf_counter(); c.load(X, y, P, eta=eta); t_load = time.perf_counter() - t0
        r = c.opt_fit_resident()          # warm-up (allocations, peer mappings)
        ts = []
        for _ in range(2):
            for d in devices:
                torch.cuda.synchronize(d)
            t0 = time.perf_counter()
            r = c.opt_fit_resident()
            ts.append(time.perf_counter() - t0)
        st = r["stats"]
        return {"workload": f"cfg3: synthetic N={N} M={M} K={K} eta={eta} fit(Opt), one process, {len(devices)} GPUs",
                "nnls_problems_per_fit": 1 << K, "s_generate": t_gen, "s_load": t_load, "s_fit_resident": float(np.mean(ts)),
                "nnls_problems_per_sec": (1 << K) / float(np.mean(ts)),
                "stages_ms": {"gram_k1_and_exchange": st["ms_gram"], "nnls_k2_k3_max_over_devices": st["ms_nnls"], "recompute_k4": st["ms_recompute"]},
                "k1_tflops_all_devices": st["gram_flops"] / (st["ms_gram"] * 1e-3) / 1e12 if st["ms_gram"] > 0 else None,
                "k2_variant": st["k2_variant"], "result": {"b_best": int(r["b_best"]), "opt": float(r["opt"])}}
    finally:
        c.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    # keep stdout clean for the one JSON line: libraries (NCCL banner, torchrun) write to fd 1 too
    json_fd = os.dup(1)
    os.dup2(2, 1)
    global _JSON_OUT
    _JSON_OUT = os.fdopen(json_fd, "w")
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
        run_native(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
