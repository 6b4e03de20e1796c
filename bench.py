#!/usr/bin/env python3
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, through libpolee_b200.so)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path on the host cores

Metric: ELBO-gradient evaluations per second (one eval = one Monte-Carlo draw's full forward+backward:
K1 SpMM + K2 transposed gradient + K3 reparameterisation/tree fwd+bwd/ADAM) on the synthetic GENCODE-scale
config C3: 30 M fragments x 200 k transcripts, nnz ~ 120 M, K = 8 draws per ADAM step.  A "step" is one ADAM
step = K evals.  At N > 1 the SAME matrix is row-partitioned into equal-nnz blocks (strong scaling) and the
transcript-length gradient is all-reduced once per step over NCCL.

value   : steady-state evals/s with the matrix resident in HBM (CUDA events on the handle's stream, max over ranks)
e2e     : the same metric through the public API with HOST buffers: one whole approximate_likelihood call
          (upload of the CSC arrays from pinned host memory, device-side layout conversion, 500 ADAM steps,
          download of mu/omega/alpha), evals / wall seconds
roofline: dominant kernel (the one-pass class kernel k_ec_lik on the default layout): algorithmic bytes (SURVEY 8d
          formula: B_K1 + B_K2, what the reference's two passes stream) / CUDA-event time vs the measured HBM peak,
          AND the bytes the kernel really moves (`moved_gbs`, `frac_moved`: the layout stores each value once, no
          indices per entry, so it moves ~6x fewer bytes than the formula charges; `frac` can therefore exceed 1)
parity  : (N = 1) lp and x_grad of one draw on the bench matrix, device vs oracle (the checker, never measured)
cpu_baseline: the oracle (C restatement of the reference's multithreaded Julia loops) on the host cores
"""
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

CONFIGS = {
    # name: (m, n, K, long_rows, seed)
    "c2": (1 << 20, 20_000, 1, False, 20260002),
    "c3": (30_000_000, 200_000, 8, False, 20260003),
    "c3-small": (3_000_000, 200_000, 8, False, 20260003),
    "c3-k6": (30_000_000, 200_000, 6, False, 20260003),   # the C3 matrix at the reference's default K (constants.jl:65)
    # C4 (heavy multi-mapping, only ever exists as per-rank blocks) and C5 (64 whole samples, one per GPU at a time):
    # see run_c4 / run_c5
    "c4": (100_000_000, 250_000, 8, True, 20260004),
    "c4-small": (8_000_000, 250_000, 8, True, 20260004),
    "c5": (30_000_000, 200_000, 8, False, 20260005),
    "c5-small": (2_000_000, 200_000, 8, False, 20260005),
}
FIT_STEPS = 500  # LIKAP_NUM_STEPS (src/constants.jl:64): what one approximate_likelihood call runs


DTYPES = {
    0: ("f32 products and in-task sums (<= 64 terms per row, <= 32 rows per lane + 5-level lane tree per column), f64 across "
        "tasks, f64 tree / ADAM arithmetic on f32 state"),
    1: ("--exact 1: f32 products summed in f64 in the reference's order (frag_probs bit-identical to the reference, split "
        "SELL + CSC kernels), f64 gradient sums, f64 tree / ADAM arithmetic on f32 state"),
    2: ("--exact 2: class kernel in f64 throughout (exact products, f64 row and column sums: at least north_star's 'fp32 "
        "with fp64 accumulation'), f64 tree / ADAM arithmetic on f32 state"),
}
DTYPE = DTYPES[0]


def workload(cfg, m, n, nnz, K):
    """config.workload: the same string in both arms."""
    return "%s: %d fragments x %d transcripts, nnz %d, K=%d draws/step, balanced-by-gene tree" % (cfg, m, n, nnz, K)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons during the timed region, sampled through NVML every few ms (the nvidia-smi
    query of B200_PROFILING.md takes longer than a whole timed region here); falls back to nvidia-smi."""

    def __init__(self, gpu_index, period_s=0.004):
        self.gpu = gpu_index
        self.period = float(os.environ.get("POLEE_BENCH_CLOCK_PERIOD_MS", period_s * 1e3)) * 1e-3
        self.sm, self.reasons = [], set()
        self.sm_max = None
        self.stop = threading.Event()
        self.t = None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # honour CUDA_VISIBLE_DEVICES: map the CUDA ordinal to the NVML device through the PCI bus id
            import torch
            bus = torch.cuda.get_device_properties(gpu_index).pci_bus_id if hasattr(
                torch.cuda.get_device_properties(gpu_index), "pci_bus_id") else None
            self.h = None
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    hh = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(hh).bus == bus:
                        self.h = hh
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _run(self):
        n = self.nvml
        bits = {}
        if n is not None:
            for name, attr in (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"),
                               ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
                               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"),
                               ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap")):
                v = getattr(n, attr, None) or getattr(n, attr.replace("ClocksEventReason", "ClocksThrottleReason"), None)
                if v is not None:
                    bits[name] = v
        while not self.stop.is_set():
            try:
                if n is not None:
                    self.sm.append(float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)))
                    get = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
                    r = get(self.h)
                    for name, b in bits.items():
                        if r & b:
                            self.reasons.add(name)
                else:
                    out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=clocks.sm,clocks.max.sm",
                                          "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                    a, b = out.strip().split(",")
                    self.sm.append(float(a)); self.sm_max = float(b)
            except Exception:
                pass
            self.stop.wait(self.period)

    def __enter__(self):
        mode = os.environ.get("POLEE_BENCH_CLOCKS", "")
        if mode == "off" or (mode == "rank0" and int(os.environ.get("RANK", "0")) != 0):
            return self
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        if self.t is not None:
            self.t.join(timeout=6)

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["unsampled"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def dump_outputs(dirname, arrays):
    """--dump-outputs: what the timed path hands its caller at the end (the fitted mu / omega / alpha), one
    DIR/<name>.npy each.  The inputs are a function of the arguments alone (seeded generator, device Philox noise
    from --seed), so two builds run with the same arguments can be compared array for array."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(dirname, name + ".npy"), a)


def generate(cfg, device):
    """Synthetic sample (polee-synth-v1) as torch tensors on `device` + host tree arrays."""
    import torch
    from polee_b200 import synth
    m, n, K, long_rows, seed = CONFIGS[cfg]
    s = synth.make_sample(m, n, seed=seed, device=device, long_rows=long_rows)
    tree = synth.balanced_tree(n, s["gene_sizes"].cpu().numpy())
    return s, tree, K


def row_block_device(s, lo, hi):
    """CSC of rows [lo, hi) (0-based) of the device-resident sample, all n columns; int32 index tensors."""
    import torch
    n = s["n"]
    rowval, nzval = s["rowval"], s["nzval"]
    if lo == 0 and hi == s["m"]:
        return hi - lo, s["colptr"].to(torch.int32), rowval.to(torch.int32), nzval
    keep = (rowval > lo) & (rowval <= hi)
    counts = torch.diff(s["colptr"])
    col_of = torch.repeat_interleave(torch.arange(n, device=rowval.device), counts)
    cnt = torch.bincount(col_of[keep], minlength=n)
    colptr = torch.cat([torch.ones(1, dtype=torch.int64, device=rowval.device), 1 + torch.cumsum(cnt, 0)])
    return hi - lo, colptr.to(torch.int32), (rowval[keep] - lo).to(torch.int32), nzval[keep].contiguous()


def equal_nnz_bounds(s, parts):
    import torch
    rows = torch.bincount(s["rowval"] - 1, minlength=s["m"])
    cum = torch.cumsum(rows, 0)
    nnz = int(cum[-1].item())
    b = [0]
    for p in range(1, parts):
        b.append(int(torch.searchsorted(cum, torch.tensor([nnz * p // parts], device=cum.device)).item()))
    b.append(s["m"])
    return b


def run_oneshot_child(args):
    """`bench.py --oneshot-child`: a fresh process that builds the same sample, makes ONE approximate_likelihood call from
    pinned host buffers and prints its wall time -- what a one-shot `polee prep-sample` pays (nothing cached on the device,
    kernels not yet loaded).  The parent bench process reports it as e2e.value."""
    import torch
    import polee_b200 as pb
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = "cuda:%d" % local
    s, tree, K = generate(args.config, dev)
    m, n = s["m"], s["n"]
    pin = lambda t, dt: torch.empty(t.shape, dtype=dt, pin_memory=True).copy_(t.to(dt)).numpy()  # noqa: E731
    colptr, rowval = pin(s["colptr"], torch.int32).view(np.uint32), pin(s["rowval"], torch.int32).view(np.uint32)
    nzval, efflens = pin(s["nzval"], torch.float32), s["efflens"].cpu().numpy()
    del s
    torch.cuda.empty_cache()
    sample = pb.RNASeqSample(m, n, colptr, rowval, nzval, efflens)
    import gc
    gc.collect()   # the generator's garbage is not part of the call
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), sample, tree_topology=tree, num_steps=FIT_STEPS,
                                    num_mc_samples=K, seed=args.seed, device=local, exact_accumulation=args.exact)
    t = time.perf_counter() - t0
    print(json.dumps({"oneshot_fit_time_s": t, "finite": bool(np.all(np.isfinite(out["mu"])))}), flush=True)


def oneshot_fit_time(args, runs=2):
    """Run run_oneshot_child in `runs` fresh processes, one after the other; returns (fastest, all times), or (None, [])
    when that is not possible (the caller then falls back to the in-process measurement).  Every run is the first call
    of a fresh process; the first process on a fresh box additionally pays for a cold file cache and driver (libraries
    read from disk, first context on the GPU), which is the box's state and not the call's cost, so the fastest stands."""
    import subprocess
    cmd = [sys.executable, os.path.abspath(__file__), "--oneshot-child", "--config", args.config, "--seed", str(args.seed),
           "--exact", str(args.exact)]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT")}
    times = []
    for _ in range(runs):
        try:
            out = subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
            if os.environ.get("POLEE_SETUP_TIMING"):   # the library's phase marks of the child, for the record
                sys.stderr.write("== one-shot child %d\n%s" % (len(times) + 1, out.stderr))
            for ln in reversed(out.stdout.splitlines()):
                if ln.startswith("{") and "oneshot_fit_time_s" in ln:
                    d = json.loads(ln)
                    if d.get("finite"):
                        times.append(float(d["oneshot_fit_time_s"]))
                    break
        except Exception:
            pass
    return (min(times), times) if times else (None, [])


def run_ours(args):
    import torch
    import torch.distributed as dist
    import polee_b200 as pb
    from polee_b200 import api as pbapi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    # The one-shot end-to-end figure comes from a fresh child process that has the GPU to itself, so it runs BEFORE this
    # process creates its CUDA context: with a second context on the device (and memory it has just freed) the child's
    # cudaMalloc calls -- 8 GB of set-up scratch -- take 140-240 ms instead of 20 (profiles/r02_cold_fit.log).
    t_oneshot, t_oneshot_all = oneshot_fit_time(args) if (world == 1 and not args.no_e2e) else (None, [])
    torch.cuda.set_device(local)
    dev = "cuda:%d" % local
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))

    s, tree, K = generate(args.config, dev)
    m, n = s["m"], s["n"]
    efflens = s["efflens"].cpu().numpy()
    nnz_total = s["nnz"]
    bounds = equal_nnz_bounds(s, world)
    m_loc, colptr_d, rowval_d, nzval_d = row_block_device(s, bounds[rank], bounds[rank + 1])
    nnz_loc = int(rowval_d.numel())

    # pinned host copies for the e2e arm: the whole matrix at N = 1 (also feeds the CPU baseline), each rank's own
    # row block at N > 1
    host = None
    pin = lambda t, dt: torch.empty(t.shape, dtype=dt, pin_memory=True).copy_(t.to(dt)).numpy()  # noqa: E731
    if not args.no_e2e:
        if world == 1:
            host = {"colptr": pin(s["colptr"], torch.int32).view(np.uint32), "rowval": pin(s["rowval"], torch.int32).view(np.uint32),
                    "nzval": pin(s["nzval"], torch.float32)}
        else:
            host = {"colptr": pin(colptr_d, torch.int32).view(np.uint32), "rowval": pin(rowval_d, torch.int32).view(np.uint32),
                    "nzval": pin(nzval_d, torch.float32)}
    # N > 1: rank 0 also fits the WHOLE matrix for 3 steps on its own (same seed => same device noise), the reference
    # point of `multi_rank_parity`
    full_params = None
    if world > 1 and rank == 0:
        hf = pb.Handle(device=local, num_mc_samples=K, num_steps=3, seed=args.seed, exact_accumulation=args.exact)
        hf.set_matrix_device(m, n, s["colptr"].to(torch.int32).data_ptr(), s["rowval"].to(torch.int32).data_ptr(),
                             s["nzval"].data_ptr())
        hf.set_efflens(efflens)
        hf.set_tree(*tree)
        hf.init_params()
        hf.run_steps(3)
        hf.sync()
        full_params = np.concatenate(hf.get_params()).astype(np.float64)
        hf.close()
    del s
    torch.cuda.empty_cache()

    h = pb.Handle(device=local, num_mc_samples=K, num_steps=max(args.steps + args.warmup, 1), seed=args.seed,
                  exact_accumulation=args.exact)
    h.set_matrix_device(m_loc, n, colptr_d.data_ptr(), rowval_d.data_ptr(), nzval_d.data_ptr())
    del colptr_d, rowval_d, nzval_d
    torch.cuda.empty_cache()
    h.set_efflens(efflens)
    h.set_tree(*tree)
    allreduce = None
    if world > 1:
        allreduce = pbapi.connect_ranks(h, dist)
    stats = h.step_stats()
    multi = None
    if world > 1:   # correctness of the row-partitioned fit, carried by the same line as its speed
        h.init_params()
        h.run_steps(3)
        h.sync()
        vec = torch.tensor(np.concatenate(h.get_params()).astype(np.float64), device=dev)
        vmax, vmin = vec.clone(), vec.clone()
        dist.all_reduce(vmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(vmin, op=dist.ReduceOp.MIN)
        multi = {"steps": 3, "identical_across_ranks": bool((vmax == vmin).all().item())}
        if rank == 0:
            multi["max_abs_param_diff_vs_single_rank"] = float(np.max(np.abs(vec.cpu().numpy() - full_params)))
            multi["what"] = ("mu/omega/alpha after 3 ADAM steps (device noise, same seed): row-partitioned over %d ranks vs "
                             "the whole matrix on rank 0 alone; the ranks differ from the single-rank fit only by the "
                             "summation order of the all-reduced gradient" % world)

    stream = torch.cuda.ExternalStream(h.stream(), device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up, then the timed region: K steps, device time on the launching stream, max over ranks
    h.init_params()
    h.run_steps(args.warmup)
    h.sync()
    # NVML inside the timed window: one query costs nothing at N = 1, but eight processes querying at once stall each
    # other's launches for milliseconds (measured: 0.81 ms/step instead of 0.29 at N = 8 with a 20-step window), so at
    # N > 1 rank 0 alone samples; the sampler is also created BEFORE the barrier (nvmlInit takes a rank-dependent time).
    if world > 1:
        os.environ.setdefault("POLEE_BENCH_CLOCKS", "rank0")
    sampler = ClockSampler(local)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with sampler as clk:
        with torch.cuda.stream(stream):
            e0.record(stream)
        h.run_steps(args.steps)
        with torch.cuda.stream(stream):
            e1.record(stream)
        h.sync()
        barrier()
    ms = e0.elapsed_time(e1)
    # before the per-kernel timings below, which launch ADAM updates of their own
    outputs = dict(zip(("mu", "omega", "alpha"), h.get_params())) if args.dump_outputs else None
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = clk.summary()
    evals_per_s = K * args.steps / (ms * 1e-3)

    # ---- per-kernel durations (CUDA events on the handle's stream, back-to-back launches; inputs >> L2)
    reps = max(5, min(50, args.steps))
    info = h.layout_info()
    t_k1, t_k2, t_k3 = (h.time_kernel(w, reps) for w in (1, 2, 3))
    t_ar = None
    if world > 1:   # the all-reduce alone, all ranks in lockstep (a rank's time includes waiting for the slowest peer)
        torch.cuda.synchronize()
        dist.barrier()
        tt = torch.tensor([h.time_kernel(5, 10)], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_ar = float(tt.item())
    peak, peak_src = measured_peak()
    # algorithmic bytes of THIS rank's launches (SURVEY 8d formula, local nnz / rows, padded draw count KP)
    KP = 1
    while KP < K:
        KP *= 2
    b_k1 = nnz_loc * 8 + (m_loc + 1) * 4 + KP * n * 4 + KP * m_loc * 4
    b_k2 = nnz_loc * 8 + (n + 1) * 4 + KP * m_loc * 4 + KP * n * 4
    onepass = stats["bytes_k2"] == 0    # one sparse pass per step: the class layout (default) or fused row tiles
    step_ms = ms / args.steps
    if onepass:
        # ONE launch does the work of the reference's two passes, so its algorithmic bytes are SURVEY 8(d)'s
        # B_K1 + B_K2 (indices + values twice + the w round trip); what it really moves is far less (`moved_gbs`,
        # `traffic`): values once, no per-entry indices, w never leaves the registers.
        if info["ec_rows"] > 0:
            kname, layout = "k_ec_lik", "equivalence classes (dense per-class blocks, one sparse pass per step)"
            t_dom = h.time_kernel(4, reps)
            share = float(info["ec_nnz"]) / max(1, nnz_loc)
            if info["general_rows"] > 0:
                layout += " + %s layout for %d rest rows" % (info["general_kind"], info["general_rows"])
        else:
            kname, layout, t_dom, share = "k12_fused_rowtiles", "fused row tiles (one sparse pass per step)", t_k1, 1.0
        achieved = share * (b_k1 + b_k2) / (t_dom * 1e-3) / 1e9
        moved = stats["bytes_k1"] / t_k1 / 1e6
        roofline = {"bound": "hbm", "kernel": kname, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                    "frac": round(achieved / peak, 4), "traffic": None, "peak_source": peak_src,
                    "note": "achieved = algorithmic bytes of K1 + K2 (SURVEY 8d; the kernel does both) / its average launch "
                            "time; moved_gbs = bytes the whole likelihood pass really streams / its time (frac_moved = "
                            "that / peak)",
                    "kernels_ms": {kname: round(t_dom, 4), "likelihood_pass_incl_second_stage": round(t_k1, 4),
                                   "k3_tree_reparam_adam": round(t_k3, 4)},
                    "kernels_gbs": {kname: round(achieved, 1)},
                    "moved_gbs": round(moved, 1), "frac_moved": round(moved / peak, 4),
                    "step_gbs": round((b_k1 + b_k2 + stats["bytes_k3"]) / step_ms / 1e6, 1),
                    "share_of_step": round(t_dom / step_ms, 3)}
        if t_ar is not None:
            roofline["kernels_ms"]["allreduce_g (max over ranks, incl. waiting for the slowest rank)"] = round(t_ar, 4)
        dom = (kname, stats["bytes_k1"], t_dom)
    else:
        layout = "split (SELL slabs for K1 + re-sorted CSC for K2)"
        dom = ("k1_sell_fwd", b_k1, t_k1) if t_k1 >= t_k2 else ("k2_csc_grad", b_k2, t_k2)
        achieved = dom[1] / (dom[2] * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom[0], "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                    "frac": round(achieved / peak, 4), "traffic": None, "peak_source": peak_src,
                    "kernels_ms": {"k1_sell_fwd": round(t_k1, 4), "k2_csc_grad": round(t_k2, 4), "k3_tree_reparam_adam": round(t_k3, 4)},
                    "kernels_gbs": {"k1_sell_fwd": round(b_k1 / t_k1 / 1e6, 1), "k2_csc_grad": round(b_k2 / t_k2 / 1e6, 1)},
                    "step_gbs": round((b_k1 + b_k2 + stats["bytes_k3"]) / step_ms / 1e6, 1),
                    "share_of_step": round(dom[2] / step_ms, 3)}
    tr = os.path.join(ROOT, "profiles", "traffic_%s.json" % args.config)
    if os.path.exists(tr) and world == 1:  # dram bytes of one launch from a committed `ncu --set full` capture (static)
        try:
            t = json.load(open(tr))
            roofline["traffic"] = t.get(dom[0])
            roofline["traffic_source"] = "static: %s" % t.get("source", "profiles/traffic_%s.json" % args.config)
        except Exception:
            pass

    # ---- parity on the bench matrix (N = 1): one draw, device vs oracle -- the oracle is the checker here
    parity = None
    xs_par = lp_par = g_par = None
    if host is not None and world == 1 and not args.no_cpu:
        xs_par = np.random.default_rng(7).dirichlet(np.ones(n)).astype(np.float32).clip(1e-10)
        lp_par, g_par = h.loglik_grad(xs_par, gradonly=False)

    # ---- e2e: one whole fit through the public API from HOST buffers
    e2e = None
    cpu = None
    if host is not None and world == 1:
        h.close()
        torch.cuda.empty_cache()
        pbapi.trim_memory(local)           # cold device allocator: what a one-shot `polee prep-sample` process sees
        sample = pb.RNASeqSample(m, n, host["colptr"], host["rowval"], host["nzval"], efflens)
        t_fits = []
        import gc
        for rep in range(2):   # [0]: cold (no cached device memory), [1]: warm (`polee prep` over many samples)
            gc.collect()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), sample, tree_topology=tree, num_steps=FIT_STEPS,
                                            num_mc_samples=K, seed=args.seed, device=local, exact_accumulation=args.exact)
            t_fits.append(time.perf_counter() - t0)
        assert np.all(np.isfinite(out["mu"]))
        h2d = host["colptr"].nbytes + host["rowval"].nbytes + host["nzval"].nbytes + efflens.nbytes + 2 * 4 * (2 * n - 1)
        # the one-shot figure: the first call of a FRESH process (nothing cached, kernels not yet loaded, CUDA graph not
        # yet built) -- what `polee prep-sample` pays.  If the child process cannot run, the first call after the
        # device-memory cache of this process was emptied stands in for it.
        t_one = t_oneshot
        t_cold = t_one if t_one is not None else t_fits[0]
        e2e = {"value": round(K * FIT_STEPS / t_cold, 1), "unit": "evals/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(3 * 4 * (n - 1)), "fit_time_s": round(t_cold, 4),
               "fit_time_source": ("first call of a fresh process that has the GPU to itself (bench.py --oneshot-child, run "
                                   "before this process creates its CUDA context); fastest of the fresh processes listed in "
                                   "oneshot_fit_times_s (the first one on a fresh box also pays for the box's cold file "
                                   "cache and driver)" if t_one is not None else
                                   "first call of this process after its device-memory cache was emptied"),
               "oneshot_fit_times_s": [round(t, 4) for t in t_oneshot_all],
               "trimmed_cache_fit_time_s": round(t_fits[0], 4),
               "warm_value": round(K * FIT_STEPS / t_fits[1], 1), "warm_fit_time_s": round(t_fits[1], 4),
               "adam_steps_per_fit": FIT_STEPS,
               "step": "one approximate_likelihood call: CSC upload from pinned host memory + device layout build + "
                       "%d ADAM steps x %d draws + parameter download; value = the one-shot call (see fit_time_source), "
                       "warm_value = a later call of the same process (cached device allocations, as in `polee prep` over "
                       "many samples)" % (FIT_STEPS, K)}
        if not args.no_cpu:
            cpu, parity = cpu_baseline(m, n, K, host, efflens, tree, budget_s=args.cpu_budget, check=(xs_par, lp_par, g_par))
    elif host is not None:
        # N > 1: every rank re-feeds its own row block from host memory into its (comm-initialised) handle and runs
        # the whole 500-step fit; wall time, max over ranks
        block = pb.RNASeqSample(m_loc, n, host["colptr"], host["rowval"], host["nzval"], efflens)
        h.opts.num_steps = FIT_STEPS
        t_fits = []
        for rep in range(2):
            barrier()
            t0 = time.perf_counter()
            h.set_sample(block)
            h.set_tree(*tree)
            h.init_params()
            h.run_steps(FIT_STEPS)
            h.sync()
            out = h.get_params()
            tt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            t_fits.append(float(tt.item()))
        h2d = host["colptr"].nbytes + host["rowval"].nbytes + host["nzval"].nbytes + efflens.nbytes + 2 * 4 * (2 * n - 1)
        hb = torch.tensor([h2d], device=dev, dtype=torch.float64)
        dist.all_reduce(hb)
        e2e = {"value": round(K * FIT_STEPS / t_fits[0], 1), "unit": "evals/s", "h2d_bytes_per_step": int(hb.item()),
               "d2h_bytes_per_step": int(3 * 4 * (n - 1)), "fit_time_s": round(t_fits[0], 4),
               "warm_value": round(K * FIT_STEPS / t_fits[1], 1), "warm_fit_time_s": round(t_fits[1], 4),
               "adam_steps_per_fit": FIT_STEPS,
               "step": "every rank: its row block's CSC upload from pinned host memory + layout build + %d ADAM steps x %d "
                       "draws (one all-reduce each) + parameter download; wall time, max over ranks; value = first call, "
                       "warm_value = second" % (FIT_STEPS, K)}
        h.close()
    else:
        h.close()
    torch.cuda.empty_cache()

    if rank == 0:
        line = {"metric": "elbo_grad_evals_per_sec", "value": round(evals_per_s, 1), "unit": "evals/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(step_ms, 4),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPES[args.exact],
                "data": "synthetic (polee-synth-v1, seed %d)" % CONFIGS[args.config][4],
                "config": {"workload": workload(args.config, m, n, nnz_total, K)},
                "details": {"partition": "rows in %d contiguous equal-nnz block(s), one per rank" % world,
                            "allreduce": ("none (one rank)" if world == 1 else
                                          "one kernel over NVLink peer memory (reduce-scatter by loads, all-gather by stores)"
                                          if allreduce == "peer" else "ncclAllReduce (Float32) between narrow / widen kernels"),
                                                        "l2": "inputs (%.2f GB/step streamed) are far larger than the 126 MB L2; no flush needed"
                                  % (stats["bytes_k1"] / 1e9 if onepass else (b_k1 + b_k2) / 1e9),
                            "layout": layout, "noise": "device Philox"},
                "clocks": clocks, "gpu_launches": int(stats["launches"] * args.steps), "roofline": roofline}
        if multi is not None:
            line["multi_rank_parity"] = multi
        if e2e:
            line["e2e"] = e2e
        if parity:
            line["parity"] = parity
        if cpu:
            line["cpu_baseline"] = cpu
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _dist_setup(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    dev = "cuda:%d" % local
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))
    return world, rank, local, dev


def run_c4(args):
    """BASELINE config 4: 100 M fragments x 250 k transcripts with heavy multi-mapping (10 % of the rows span 64-512
    transcripts), row-partitioned over the ranks with one NCCL all-reduce per step.  The matrix never exists as a whole:
    every rank generates its own block of m / N rows on its GPU (same transcriptome, its own rows: synth row_seed)."""
    import torch
    import torch.distributed as dist
    import polee_b200 as pb
    from polee_b200 import api as pbapi, synth
    world, rank, local, dev = _dist_setup(args)
    m, n, K, long_rows, seed = CONFIGS[args.config]
    m_loc = m // world
    if m_loc * 40 > 2**31 - 1:
        raise SystemExit("%s needs more ranks: %d rows per rank would exceed 2^31 entries" % (args.config, m_loc))
    s = synth.make_sample(m_loc, n, seed=seed, device=dev, long_rows=True, row_seed=seed * 1000 + rank)
    tree = synth.balanced_tree(n, s["gene_sizes"].cpu().numpy())
    efflens = s["efflens"].cpu().numpy()
    nnz_loc = s["nnz"]
    colptr_d, rowval_d, nzval_d = s["colptr"].to(torch.int32), s["rowval"].to(torch.int32), s["nzval"]
    del s
    torch.cuda.empty_cache()
    h = pb.Handle(device=local, num_mc_samples=K, num_steps=max(args.steps + args.warmup, 1), seed=args.seed)
    t0 = time.perf_counter()
    h.set_matrix_device(m_loc, n, colptr_d.data_ptr(), rowval_d.data_ptr(), nzval_d.data_ptr())
    torch.cuda.synchronize()
    t_layout = time.perf_counter() - t0
    del colptr_d, rowval_d, nzval_d
    torch.cuda.empty_cache()
    h.set_efflens(efflens)
    h.set_tree(*tree)
    allreduce = None
    if world > 1:
        allreduce = pbapi.connect_ranks(h, dist)
        os.environ.setdefault("POLEE_BENCH_CLOCKS", "rank0")
    stats, info = h.step_stats(), h.layout_info()
    stream = torch.cuda.ExternalStream(h.stream(), device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    h.init_params()
    h.run_steps(args.warmup)
    h.sync()
    sampler = ClockSampler(local)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with sampler as clk:
        e0.record(stream)
        h.run_steps(args.steps)
        e1.record(stream)
        h.sync()
        barrier()
    ms = e0.elapsed_time(e1)
    tot = torch.tensor([float(nnz_loc), float(info["ec_nnz"]), float(info["general_nnz"])], device=dev, dtype=torch.float64)
    tmax = torch.tensor([ms, t_layout], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tot)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms, t_layout = float(tmax[0].item()), float(tmax[1].item())
    out = h.get_params()
    finite = bool(all(np.all(np.isfinite(v)) for v in out))
    reps = max(5, min(20, args.steps))
    t_k1, t_k2, t_k3 = (h.time_kernel(w, reps) for w in (1, 2, 3))
    t_ec = h.time_kernel(4, reps) if info["ec_rows"] > 0 else 0.0
    peak, peak_src = measured_peak()
    KP = 8
    gm, gnnz = info["general_rows"], info["general_nnz"]
    b_k1 = gnnz * 8 + (gm + 1) * 4 + KP * n * 4 + KP * gm * 4      # the general (split) layout's two passes: SURVEY 8d
    b_k2 = gnnz * 8 + (n + 1) * 4 + KP * gm * 4 + KP * n * 4
    h.close()
    if rank == 0:
        nnz_total = int(tot[0].item())
        # dominant kernel: the long rows (> 64 transcripts) take the general split layout; K2 of it streams the most
        cand = {"k1_sell_fwd": (b_k1, t_k1 - t_ec - 0.0), "k2_csc_grad": (b_k2, t_k2)}
        if t_k2 <= 0:   # fused / class-only layouts: report the whole pass
            cand = {"likelihood_pass": (stats["bytes_k1"], t_k1)}
        kname = max(cand, key=lambda k: cand[k][1])
        ach = cand[kname][0] / max(cand[kname][1], 1e-9) / 1e6
        line = {"metric": "elbo_grad_evals_per_sec", "value": round(K * args.steps / (ms * 1e-3), 1), "unit": "evals/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 4),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE,
                "data": "synthetic (polee-synth-v1, seed %d; every rank generates its own row block on its GPU)" % seed,
                "config": {"workload": workload(args.config, m_loc * world, n, nnz_total, K)},
                "details": {"partition": "%d ranks x %d rows each (same transcriptome, independent rows)" % (world, m_loc),
                            "allreduce": ("none (one rank)" if world == 1 else
                                          "one kernel over NVLink peer memory (reduce-scatter by loads, all-gather by stores)"
                                          if allreduce == "peer" else "ncclAllReduce (Float32) between narrow / widen kernels"),
                                                        "layout": "class layout: %.1f %% of the entries; general %s layout (rows longer than 64 "
                                      "transcripts): %.1f %%" % (100 * tot[1].item() / nnz_total, info["general_kind"],
                                                                 100 * tot[2].item() / nnz_total),
                            "layout_build_s": round(t_layout, 3), "finite_fit": finite,
                            "e2e": "not run: the per-rank blocks (%.1f GB of CSC each) are generated on the device"
                                   % (nnz_loc * 8 / 1e9)},
                "clocks": clk.summary(), "gpu_launches": int(stats["launches"] * args.steps),
                "roofline": {"bound": "hbm", "kernel": kname, "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                             "frac": round(ach / peak, 4), "traffic": None, "peak_source": peak_src,
                             "kernels_ms": {"likelihood_pass_class+k1": round(t_k1, 4), "k_ec_lik": round(t_ec, 4),
                                            "k2_csc_grad": round(t_k2, 4), "k3_tree_reparam_adam": round(t_k3, 4)},
                             "note": "rank 0's launches; bytes = SURVEY 8(d) formula on the rows of the general layout"}}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dict(zip(("mu", "omega", "alpha"), out)))
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_c5(args):
    """BASELINE config 5: batch prep of 64 GTEx-shaped samples, whole samples per GPU (replicas only, no collective;
    src/main.jl:590-631 is the loop).  Every rank fits its share of the samples one after another through the public
    API from pinned HOST buffers (upload + layout build + 500 ADAM steps + download); a sample's synthetic generation
    (which stands in for the reference's BAM parsing) is outside the timed sum.  value = aggregate evals/s."""
    import torch
    import torch.distributed as dist
    import polee_b200 as pb
    from polee_b200 import synth
    world, rank, local, dev = _dist_setup(args)
    m0, n, K, _, seed = CONFIGS[args.config]
    n_samples = args.samples
    rng = np.random.default_rng(seed)
    sizes = np.clip(m0 * np.exp(0.35 * rng.standard_normal(n_samples)), m0 / 2, m0 * 2).astype(np.int64)  # depth spread +-2x
    mine = list(range(rank, n_samples, world))
    pin = lambda t, dt: torch.empty(t.shape, dtype=dt, pin_memory=True).copy_(t.to(dt)).numpy()  # noqa: E731
    t_sum, evals, h2d, nnz_sum = 0.0, 0, 0, 0
    fits = []
    with ClockSampler(local, period_s=0.05) as clk:
        for i in mine:
            s = synth.make_sample(int(sizes[i]), n, seed=seed + 1 + i, device=dev)
            tree = synth.balanced_tree(n, s["gene_sizes"].cpu().numpy())
            host = {"colptr": pin(s["colptr"], torch.int32).view(np.uint32), "rowval": pin(s["rowval"], torch.int32).view(np.uint32),
                    "nzval": pin(s["nzval"], torch.float32)}
            efflens = s["efflens"].cpu().numpy()
            nnz_sum += s["nnz"]
            del s
            torch.cuda.empty_cache()
            sample = pb.RNASeqSample(int(sizes[i]), n, host["colptr"], host["rowval"], host["nzval"], efflens)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = pb.approximate_likelihood(pb.LogitSkewNormalPTTApprox(), sample, tree_topology=tree, num_steps=FIT_STEPS,
                                            num_mc_samples=K, seed=args.seed + i, device=local)
            dt = time.perf_counter() - t0
            assert np.all(np.isfinite(out["mu"]))
            fits.append(dt)
            t_sum += dt
            evals += K * FIT_STEPS
            h2d += host["colptr"].nbytes + host["rowval"].nbytes + host["nzval"].nbytes + efflens.nbytes + 2 * 4 * (2 * n - 1)
    agg = torch.tensor([float(evals), float(h2d), float(nnz_sum), float(len(mine))], device=dev, dtype=torch.float64)
    tmax = torch.tensor([t_sum], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(agg)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    T = float(tmax.item())
    if rank == 0:
        v = agg[0].item() / T
        line = {"metric": "elbo_grad_evals_per_sec", "value": round(v, 1), "unit": "evals/s", "n_gpus": world,
                "steps": FIT_STEPS, "warmup": 0, "ms_per_step": round(T / (len(mine) * FIT_STEPS) * 1e3, 4),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
                "data": "synthetic (polee-synth-v1, seeds %d..%d)" % (seed + 1, seed + n_samples),
                "config": {"workload": "%s: %d samples, m ~ LogNormal around %d (x0.5..x2), %d transcripts, K=%d, %d ADAM steps "
                                       "each; whole samples per GPU, no collective" % (args.config, n_samples, m0, n, K, FIT_STEPS)},
                "details": {"samples_per_s": round(agg[3].item() / T, 3), "job_time_s": round(T, 3),
                            "rank0_fit_times_s": [round(x, 3) for x in fits], "total_nnz": int(agg[2].item()),
                            "timed": "sum over a rank's samples of the approximate_likelihood wall time from pinned host "
                                     "buffers (upload, layout build, fit, download); max over ranks"},
                "clocks": clk.summary(), "gpu_launches": None,
                "e2e": {"value": round(v, 1), "unit": "evals/s", "h2d_bytes_per_step": int(agg[1].item() / agg[3].item()),
                        "d2h_bytes_per_step": int(3 * 4 * (n - 1)),
                        "step": "here a step = one whole sample (the e2e path IS the measured path of this config)"}}
        if args.dump_outputs and fits:   # the fit of rank 0's last sample
            dump_outputs(args.dump_outputs, {k: out[k] for k in ("mu", "omega", "alpha")})
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def cpu_baseline(m, n, K, host, efflens, tree, budget_s=25.0, warm=0, check=None):
    """The oracle (C/OpenMP restatement of the reference's Julia loops) on the host cores: whole ADAM steps of
    K draws on the SAME matrix, as many as fit in the budget (at least one).  With check = (xs, lp, x_grad) of one
    device evaluation it also returns the parity block (device vs oracle on that draw)."""
    from oracle import polee_oracle as O
    O.set_num_threads()   # all cores (the reference's wrapper policy, polee:8-12), whatever OMP_NUM_THREADS says
    parity = None
    if check is not None and check[0] is not None:
        xs, lp_d, g_d = check
        lp_o, g_o = O.Model(m, n, host["colptr"], host["rowval"], host["nzval"]).log_likelihood(xs, gradonly=False)
        nz = g_o != 0
        parity = {"lp_relerr": float(abs(lp_d[0] - lp_o) / abs(lp_o)),
                  "x_grad_relerr": float(np.max(np.abs(g_d[0][nz] - g_o[nz]) / g_o[nz])),
                  "zero_columns_equal": bool(np.array_equal(g_d[0][~nz], g_o[~nz])), "tolerance": 1e-5,
                  "what": "one draw x ~ Dirichlet(1) on the bench matrix: device loglik_grad (default arithmetic) vs the "
                          "oracle (Float32 products, Float64 sums in the reference's order); max over the non-empty columns"}
    st = O.FitStepper(m, n, host["colptr"], host["rowval"], host["nzval"], efflens, tree[0], tree[1], num_mc_samples=K)
    for _ in range(warm):
        st.step()
    t0 = time.perf_counter()
    steps = 0
    while True:
        st.step()
        steps += 1
        el = time.perf_counter() - t0
        if el > budget_s or el + el / steps > budget_s * 1.3:
            break
    st.close()
    return {"value": round(K * steps / el, 3), "unit": "evals/s", "cores": O.num_threads(), "kind": "port",
            "sample": "%d full ADAM step(s) of %d draws on the same %d x %d matrix (setup/transposition excluded), "
                      "%.1f s" % (steps, K, m, n, el)}, parity


def run_reference(args):
    """Reference arm: the reference's CPU algorithm (oracle port -- Julia is not installable here) with all host
    threads, same config/metric.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    from polee_b200 import synth
    m, n, K, long_rows, seed = CONFIGS[args.config]
    dev = "cuda:0" if torch.cuda.is_available() else "cpu"
    scale, scale_note = 1.0, ""
    if args.config.startswith("c4"):
        # the whole C4 matrix does not fit the host: time the block of ONE of 8 ranks (1/8 of the rows, the same
        # generator the GPU arm uses) and divide -- every loop of the path is linear in the rows
        parts = 8
        s = synth.make_sample(m // parts, n, seed=seed, device=dev, long_rows=True, row_seed=seed * 1000)
        scale, scale_note = 1.0 / parts, "; timed on 1/%d of the rows (one rank's block), value = that / %d" % (parts, parts)
    elif args.config.startswith("c5"):
        s = synth.make_sample(m, n, seed=seed + 1, device=dev)   # one sample of the median size: samples are sequential on a CPU
        scale_note = "; one median-size sample (the CPU fits samples one after another, so evals/s is per sample)"
    else:
        s = synth.make_sample(m, n, seed=seed, device=dev, long_rows=long_rows)
    m = s["m"]
    tree = synth.balanced_tree(n, s["gene_sizes"].cpu().numpy())
    ns = synth.to_numpy_sample(s)
    nnz = s["nnz"]
    del s
    from oracle import polee_oracle as O
    cores = O.set_num_threads()   # all cores: torch.distributed.run exports OMP_NUM_THREADS=1
    st = O.FitStepper(m, n, ns["colptr"], ns["rowval"], ns["nzval"], ns["efflens"], tree[0], tree[1], num_mc_samples=K)
    budget = args.cpu_budget * 4
    t_w = time.perf_counter()
    done_w = 0
    for _ in range(args.warmup):
        st.step()
        done_w += 1
        if time.perf_counter() - t_w > budget / 4:
            break
    t0 = time.perf_counter()
    steps = 0
    for _ in range(args.steps):
        st.step()
        steps += 1
        if args.budget_steps and time.perf_counter() - t0 > budget:
            break
    el = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("mu", "omega", "alpha"), st.params())))
    st.close()
    v = round(K * steps / el * scale, 3)
    within = "within a %.0f s budget" % budget if args.budget_steps else "(--steps: no time budget)"
    sample = "%d of the %d requested ADAM steps (x %d draws) on the full matrix %s; %d warm-up%s" % (
        steps, args.steps, K, within, done_w, scale_note)
    print(json.dumps({
        "impl": "reference", "metric": "elbo_grad_evals_per_sec", "value": v, "unit": "evals/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": done_w, "ms_per_step": round(el / steps * 1e3, 2), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32 products, f64 sums (the reference's arithmetic)",
        "data": "synthetic (polee-synth-v1, seed %d)" % seed,
        "config": {"workload": workload(args.config, m, n, nnz, K)},
        "details": {"note": "CPU restatement of the reference's multithreaded Julia path (oracle/polee_oracle.c, OpenMP "
                            "static chunks = Threads.@threads) on %d threads; Julia itself is not available" % cores},
        "cpu_baseline": {"value": v, "unit": "evals/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 50)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS))
    ap.add_argument("--seed", type=int, default=123456789)
    ap.add_argument("--exact", type=int, default=0, choices=[0, 1, 2],
                    help="opts.exact_accumulation: 0 default arithmetic, 1 reference-order Float64 accumulation (split kernels), "
                         "2 class kernel in Float64")
    ap.add_argument("--oneshot-child", action="store_true", help="internal: one fit in this fresh process, print its time")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=25.0)
    ap.add_argument("--samples", type=int, default=64, help="c5: number of samples")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the fitted mu / omega / alpha as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.steps is not None and args.config.startswith("c5"):
        ap.error("--steps does not apply to %s: every sample is one whole %d-step fit" % (args.config, FIT_STEPS))
    # the reference arm stops at its time budget only when the number of steps was left to it
    args.budget_steps = args.steps is None
    args.steps = 50 if args.steps is None else args.steps
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.oneshot_child:
        run_oneshot_child(args)
    elif args.impl == "reference":
        run_reference(args)
    elif args.config.startswith("c4"):
        run_c4(args)
    elif args.config.startswith("c5"):
        run_c5(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
