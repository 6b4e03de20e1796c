"""Kernel durations and the idle gaps between them in the steady-state ADAM step loop (graph-replayed, as bench.py times
it), from a torch.profiler trace with CUDA activities.

    python tools/step_gaps.py [--config c3] [--warmup 10] [--steps 24] [--trace DIR]
    python tools/step_gaps.py --from-trace FILE      # the tables of a trace this tool wrote earlier

For every kernel of the step's main chain it prints the median duration over the traced steps and the median idle gap
before it: the start of the kernel minus the end of the chain kernel before it.  A negative gap is an overlap (a
programmatically launched kernel started while its predecessor drained); a kernel's duration then includes the time
its CTAs spent waiting for the predecessor.  The side-stream kernel (k3_leaf_S, or k3_mid) is listed with its duration
only.  The chain is told apart by kernel name, not by stream: a replayed graph spreads its kernels over streams of its
own.  The step period is the distance between the starts of consecutive tree-forward kernels.

POLEE_PDL is read from the environment when the handle is created, so `POLEE_PDL=0 python tools/step_gaps.py` and
`POLEE_PDL=1 ...` in one job compare both launch modes of one build.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np


def short_name(name):
    """`void polee::(anonymous namespace)::k_ec_lik<float, 8, false>(...)` -> `k_ec_lik<float, 8, false>`"""
    name = re.sub(r"^void\s+", "", name).replace("(anonymous namespace)::", "")
    head, sep, tail = name.split("(")[0].partition("<")
    return head.split("::")[-1] + sep + tail


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c3")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--steps", type=int, default=24, help="traced steps (the first and last are dropped)")
    ap.add_argument("--trace", default=None, help="directory for the chrome trace (default: a temporary one)")
    ap.add_argument("--from-trace", default=None, help="print the tables of an existing trace instead of running")
    a = ap.parse_args()
    if a.from_trace:
        report(a.from_trace, "trace %s" % a.from_trace)
        return

    import torch
    from torch.profiler import ProfilerActivity, profile
    import polee_b200 as pb
    from bench import generate, row_block_device

    torch.cuda.set_device(0)
    s, tree, K = generate(a.config, "cuda:0")
    m, n = s["m"], s["n"]
    _, colptr, rowval, nzval = row_block_device(s, 0, m)
    h = pb.Handle(device=0, num_mc_samples=K, num_steps=a.warmup + a.steps)
    h.set_matrix_device(m, n, colptr.data_ptr(), rowval.data_ptr(), nzval.data_ptr())
    h.set_efflens(s["efflens"].cpu().numpy())
    h.set_tree(*tree)
    del s, colptr, rowval, nzval
    torch.cuda.empty_cache()
    h.init_params()
    h.run_steps(a.warmup)
    h.sync()
    torch.cuda.synchronize()

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        h.run_steps(a.steps)
        h.sync()
        torch.cuda.synchronize()
    tdir = a.trace or tempfile.mkdtemp(prefix="step_gaps_")
    os.makedirs(tdir, exist_ok=True)
    path = os.path.join(tdir, "step_gaps_pdl%s.json" % os.environ.get("POLEE_PDL", "default"))
    prof.export_chrome_trace(path)
    info = h.layout_info()
    h.close()
    report(path, "card: %s | config %s | POLEE_PDL=%s | %d traced steps after %d warm-up steps\n"
           "programmatic edges of the captured graphs: one-step %d, multi-step %d"
           % (card(), a.config, os.environ.get("POLEE_PDL", "(unset)"), a.steps, a.warmup,
              info["graph_programmatic_edges"], info["multi_step_graph_programmatic_edges"]))


def report(path, header):
    ev = [e for e in json.load(open(path))["traceEvents"] if e.get("cat") == "kernel"]
    ev.sort(key=lambda e: e["ts"])
    side_names = ("k3_leaf_S", "k3_mid")
    mev = [e for e in ev if not short_name(e["name"]).startswith(side_names)]
    starts = [i for i, e in enumerate(mev) if "tree_fwd" in e["name"]]
    # whole steps only, without the first (graph launch from an idle stream) and the last
    steps = [mev[starts[j]:starts[j + 1]] for j in range(1, len(starts) - 1)]
    prev_end = {id(e): (mev[i - 1]["ts"] + mev[i - 1]["dur"]) if i else None for i, e in enumerate(mev)}
    order, dur, gap = [], {}, {}
    for st in steps:
        seen = {}
        for e in st:
            nm = short_name(e["name"])
            seen[nm] = seen.get(nm, 0) + 1
            key = nm if seen[nm] == 1 else "%s #%d" % (nm, seen[nm])
            if key not in dur:
                order.append(key)
                dur[key], gap[key] = [], []
            dur[key].append(e["dur"])
            gap[key].append(e["ts"] - prev_end[id(e)])
    period = [mev[starts[j + 1]]["ts"] - mev[starts[j]]["ts"] for j in range(1, len(starts) - 1)]
    side = {}
    for e in ev:
        if short_name(e["name"]).startswith(side_names):
            side.setdefault(short_name(e["name"]), []).append(e["dur"])

    print(header)
    print("%d whole steps in the table" % len(steps))
    print("%-44s %12s %14s" % ("step kernel (main chain)", "median us", "gap before us"))
    tot_gap = 0.0
    for key in order:
        g = float(np.median(gap[key]))
        tot_gap += g
        print("%-44s %12.2f %14.2f" % (key[:44], float(np.median(dur[key])), g))
    for nm, d in side.items():
        print("%-44s %12.2f %14s" % (("[side] " + nm)[:44], float(np.median(d)), "-"))
    print("sum of median gaps per step: %.2f us" % tot_gap)
    print("step period (tree-forward start to start): median %.2f us, min %.2f, max %.2f"
          % (float(np.median(period)), min(period), max(period)))
    print("trace: %s" % path)


if __name__ == "__main__":
    main()
