#!/usr/bin/env python3
"""K5 measurement: log q(x) of the LogitSkewNormalPTT approximation (polee_approx_log_prob_device) for B = 64 rows of
n = 200 000 transcripts, parameters per row, shared tree and a tree per row (the synth trees of tools/bench_hsb.py),
device buffers on a stream, CUDA events after warm-up.  Next to it, on the same plan and inputs, the composition a
caller has without the op: inv_hsb_device -> torch Float64 elementwise ops for the LSN terms -> inv_hsb_grad_device.

    python tools/bench_approx_log_prob.py [--B 64] [--n 200000] [--reps 20] [--rounds 3]
Prints the card (name, power limit), then one JSON line per (tree mode, variant): median over rounds of the mean time
of `reps` back-to-back calls, algorithmic bytes (x, parameters and index arrays read once, lp and x_grad written
once) and the rate they give.  The working set (~0.6 GB of inputs and scratch) is far larger than the 126 MB L2."""
import argparse
import json
import math
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import polee_b200 as pb  # noqa: E402
from polee_b200 import synth  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout
        name, power = [s.strip() for s in out.strip().splitlines()[0].split(",")]
    except Exception as e:  # the timings stand without it, but say so
        name, power = "unknown (%s)" % e, "unknown"
    return {"card": name, "power_limit": power}


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=64)
    ap.add_argument("--n", type=int, default=200000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    B, n, N = a.B, a.n, 2 * a.n - 1
    print(json.dumps(card()), flush=True)
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(0)
    t = lambda v, dt=torch.float32: torch.from_numpy(np.ascontiguousarray(v)).to(dev, dt)  # noqa: E731
    mu = t(rng.uniform(-2, 2, (B, n - 1)))
    omega = t(np.log(rng.uniform(0.1, 1.0, (B, n - 1))))
    alpha = t(rng.uniform(-0.5, 0.5, (B, n - 1)))
    z0 = torch.from_numpy(rng.normal(size=(B, n - 1))).to(dev)
    y_logit = (mu.double() + torch.exp(omega).double() * torch.sinh(alpha.double() + torch.asinh(z0))).float()
    l, r, f = pb.make_inverse_ptt_params(*synth.balanced_tree(n))
    st = torch.cuda.Stream()
    S = st.cuda_stream
    for mode in ("shared", "per_row"):
        ib = 1 if mode == "shared" else B
        plan = pb.HsbPlan(n, *(np.ascontiguousarray(np.broadcast_to(v, (ib, N))) for v in (l, r, f)))
        with torch.cuda.stream(st):
            x = torch.empty((B, n), dtype=torch.float32, device=dev)
            plan.hsb_device(B, y_logit.data_ptr(), x.data_ptr(), S)        # x on the simplex, drawn from q
            lp = torch.empty(B, dtype=torch.float64, device=dev)
            x_grad = torch.empty((B, n), dtype=torch.float32, device=dev)
            y = torch.empty((B, n - 1), dtype=torch.float64, device=dev)
            ladj = torch.empty((B, 1), dtype=torch.float32, device=dev)
            ones = torch.ones((B, 1), dtype=torch.float32, device=dev)
            c_grad = torch.empty((B, n), dtype=torch.float32, device=dev)
        out = {}

        def op(grad):
            plan.approx_log_prob_device(B, B, x.data_ptr(), mu.data_ptr(), omega.data_ptr(), alpha.data_ptr(),
                                        lp.data_ptr(), x_grad.data_ptr() if grad else 0, S)

        def composition(grad):
            plan.inv_hsb_device(B, x.data_ptr(), y.data_ptr(), ladj.data_ptr(), S)
            with torch.cuda.stream(st):
                sigma = torch.exp(omega).double()
                ly, l1my = torch.log(y), torch.log1p(-y)
                s = (ly - l1my - mu.double()) / sigma
                w = torch.asinh(s) - alpha.double()
                z0, aw = torch.sinh(w), w.abs()
                term = (-0.5 * z0 * z0 - 0.5 * math.log(2 * math.pi) + aw + torch.log1p(torch.exp(-2.0 * aw)) - math.log(2.0)
                        - 0.5 * torch.log1p(s * s) - torch.log(sigma) - ly - l1my)
                out["lp"] = term.sum(1) + ladj[:, 0].double()
                if grad:
                    rr = torch.hypot(torch.ones_like(s), s)
                    g_s = (torch.tanh(w) - z0 * torch.cosh(w)) / rr - s / (rr * rr)
                    y_grad = (g_s / (sigma * y * (1.0 - y)) + 1.0 / (1.0 - y) - 1.0 / y).contiguous()
                    out["y_grad"] = y_grad
            if grad:
                plan.inv_hsb_grad_device(B, out["y_grad"].data_ptr(), ones.data_ptr(), y.data_ptr(), c_grad.data_ptr(), S)

        def timed(fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(a.reps):
                fn()
            e1.record(st)
            st.synchronize()
            return e0.elapsed_time(e1) / a.reps

        variants = {"op_lp": lambda: op(False), "op_lp_grad": lambda: op(True),
                    "composition_lp": lambda: composition(False), "composition_lp_grad": lambda: composition(True)}
        for fn in variants.values():   # warm-up: module loads, plan scratch, torch's allocator
            fn(); fn()
        st.synchronize()
        times = {k: [] for k in variants}
        for _ in range(a.rounds):      # alternate the variants inside each round
            for k, fn in variants.items():
                times[k].append(timed(fn))
        # the two paths agree: lp up to the composition's Float32 ladj, x_grad up to Float32 rounding
        op(True)
        composition(True)
        st.synchronize()
        lp_rel = ((out["lp"] - lp).abs() / lp.abs()).max().item()
        g_rel = ((c_grad - x_grad).abs().amax(1) / x_grad.abs().amax(1)).max().item()
        idx_bytes = ib * N * 12
        base = B * n * 4 + 3 * B * (n - 1) * 4 + idx_bytes + B * 8
        for k, ts in times.items():
            ms = float(np.median(ts))
            alg = base + (B * n * 4 if k.endswith("grad") else 0)
            print(json.dumps({"op": "approx_log_prob", "variant": k, "trees": mode, "B": B, "n": n, "param_batch": B,
                              "ms": round(ms, 4), "ms_rounds": [round(v, 4) for v in ts], "algorithmic_GB": round(alg / 1e9, 4),
                              "GBps": round(alg / (ms * 1e-3) / 1e9, 1), "reps": a.reps,
                              "max_rel_lp_vs_composition": lp_rel, "max_rel_xgrad_vs_composition": g_rel}), flush=True)
        plan.close()


if __name__ == "__main__":
    main()
