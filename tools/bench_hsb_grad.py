#!/usr/bin/env python3
"""HSBGrad measurement (DESIGN.md K4) at B = 64 rows x n = 200 000 leaves, a shared balanced tree and a tree per row
(the balanced tree with its leaves permuted differently in every row), next to HSB (polee_hsb_device) on the same plan.

Device-resident form (polee_hsb_grad_device): CUDA events around `--calls` back-to-back calls on one stream after a
warm-up; the mean per call, and the median of `--rounds` rounds.  The inputs (x_grad and y_logit, 102 MB at the default
size) plus the output do not fit the 126 MB L2.  Host-buffer form (polee_hsb_grad_with_plan): wall clock per call,
including the PCIe copies.  Bytes per call are SURVEY 8(d)'s K4 formula extended to HSBGrad:
B n 4 (x_grad) + 2 B (n - 1) 4 (y_logit in, gradient out) + 12 (2n - 1) per distinct tree (left, right, leaf).

    python tools/bench_hsb_grad.py [--B 64] [--n 200000] [--out profiles/FILE.jsonl]
Prints one JSON line per (tree mode, op, form), with the card's name and power limit."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import polee_b200 as pb  # noqa: E402
from polee_b200 import _lib as L, synth  # noqa: E402

P = C.c_void_p
p = lambda a: a.ctypes.data_as(P)  # noqa: E731


def card():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = (s.strip() for s in q.split(","))
    except Exception as e:  # the measurement stands without it, but says so
        out["power_limit"] = "unknown (%s)" % e
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=64)
    ap.add_argument("--n", type=int, default=200000)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--host-calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    B, n, N = a.B, a.n, 2 * a.n - 1
    lib = L.load_library()
    info = card()
    rng = np.random.default_rng(0)
    lines = []
    pi, js = synth.balanced_tree(n)
    for mode in ("shared", "per_row"):
        if mode == "shared":
            idx = [v[None] for v in pb.make_inverse_ptt_params(pi, js)]
        else:
            rows = []
            for _ in range(B):
                perm = np.concatenate([[0], rng.permutation(n) + 1]).astype(np.int32)
                rows.append(pb.make_inverse_ptt_params(pi, np.where(js > 0, perm[js], 0).astype(np.int32)))
            idx = [np.ascontiguousarray(np.stack(v)) for v in zip(*rows)]
        ib = idx[0].shape[0]
        plan = pb.HsbPlan(n, *idx)
        x_grad = rng.normal(size=(B, n)).astype(np.float32)
        y_logit = rng.normal(0, 2, (B, n - 1)).astype(np.float32)
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            d_xg, d_yl = torch.from_numpy(x_grad).cuda(), torch.from_numpy(y_logit).cuda()
            d_out = torch.empty((B, n - 1), dtype=torch.float32, device="cuda")
            d_x = torch.empty((B, n), dtype=torch.float32, device="cuda")
        st.synchronize()
        S = st.cuda_stream
        ops = {"hsb_grad": lambda: plan.hsb_grad_device(B, d_xg.data_ptr(), d_yl.data_ptr(), d_out.data_ptr(), S),
               "hsb": lambda: plan.hsb_device(B, d_yl.data_ptr(), d_x.data_ptr(), S)}

        def dev_round(fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(a.calls):
                fn()
            e1.record(st)
            st.synchronize()
            return e0.elapsed_time(e1) / a.calls

        for fn in ops.values():  # warm-up
            fn(); fn()
        st.synchronize()
        ms = {k: [] for k in ops}
        for _ in range(a.rounds):  # the ops alternate round by round
            for k, fn in ops.items():
                ms[k].append(dev_round(fn))
        host_out = np.zeros((B, n - 1), np.float32)
        lib.polee_hsb_grad_with_plan(plan.p, C.c_int64(B), p(x_grad), p(y_logit), p(host_out))
        host = []
        for _ in range(a.host_calls):
            t = time.perf_counter()
            assert lib.polee_hsb_grad_with_plan(plan.p, C.c_int64(B), p(x_grad), p(y_logit), p(host_out)) == 0
            host.append((time.perf_counter() - t) * 1e3)
        assert np.array_equal(d_out.cpu().numpy(), host_out)
        idx_bytes = ib * N * 12
        alg = {"hsb_grad": B * n * 4 + 2 * B * (n - 1) * 4 + idx_bytes, "hsb": B * (n - 1) * 4 + B * n * 4 + idx_bytes}
        for op in ops:
            t = statistics.median(ms[op])
            lines.append({"op": op, "form": "device_resident", "trees": mode, "B": B, "n": n, "ms": round(t, 4),
                          "rounds_ms": [round(v, 4) for v in ms[op]], "calls_per_round": a.calls,
                          "algorithmic_GB": round(alg[op] / 1e9, 4), "GBps": round(alg[op] / t / 1e6, 1), **info})
        t = statistics.median(host)
        lines.append({"op": "hsb_grad", "form": "host_buffers", "trees": mode, "B": B, "n": n, "ms": round(t, 2),
                      "calls": a.host_calls, "GBps_incl_pcie": round(alg["hsb_grad"] / t / 1e6, 1), **info})
        plan.close()
    for ln in lines:
        print(json.dumps(ln))
    if a.out:
        with open(a.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
