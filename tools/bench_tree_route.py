"""Time the K3 group (polee_time_kernel(3): tree forward, S, tree backward, update + reparameterisation) on a tree that
takes the shared-memory level kernels (route "levels_smem"): synth.spine_tree, deep and not in a shape the DFS-run,
path-product or chain kernels serve.  Prints one JSON line.  POLEE_B200_LIB times another build of the library, so that
two builds can be compared in one session, alternating."""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import polee_b200 as pb  # noqa: E402
from polee_b200 import synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--spine", type=int, default=1200, help="internal nodes on the spine")
ap.add_argument("--every", type=int, default=100, help="a 3-leaf subtree every this many spine nodes")
ap.add_argument("--K", type=int, default=6, help="draws per step")
ap.add_argument("--reps", type=int, default=200, help="launches of the group per measurement")
ap.add_argument("--repeat", type=int, default=7, help="measurements (the median is reported)")
a = ap.parse_args()

pi, js = synth.spine_tree(a.spine, a.every)
n = (len(pi) + 1) // 2
s = synth.to_numpy_sample(synth.make_sample(20 * n, n, seed=7))
h = pb.Handle(num_mc_samples=a.K)
h.set_sample(pb.RNASeqSample(s["m"], s["n"], s["colptr"], s["rowval"], s["nzval"], s["efflens"]), tree_topology=(pi, js))
h.time_kernel(3, 20)  # loads the kernels, sizes the work buffers
ms = [h.time_kernel(3, a.reps) for _ in range(a.repeat)]
print(json.dumps({"tree": "spine_tree(%d, %d)" % (a.spine, a.every), "n": n, "K": a.K,
                  "tree_route": h.layout_info()["tree_route"], "lib": os.environ.get("POLEE_B200_LIB", "in-tree"),
                  "k3_ms_median": statistics.median(ms), "k3_ms_min": min(ms), "k3_ms_max": max(ms)}))
h.close()
