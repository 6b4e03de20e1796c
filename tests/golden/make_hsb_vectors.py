#!/usr/bin/env python3
"""Golden vectors for the three HSB ops, produced by the REFERENCE's own code.

Runs the reference's src/tensorflow_ext/hsb_ops.cpp -- compiled unmodified into oracle/_ref/ over the stub
TF API (oracle/Makefile target `ref`) -- on seeded inputs and stores inputs + outputs.  It needs a checkout of
the original Polee; the .npz is committed so that the tests need none.

    python tests/golden/make_hsb_vectors.py <polee checkout>
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import polee_oracle as O  # noqa: E402
from polee_b200 import synth  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")


def main(reference):
    O.build(force=True, reference=reference)   # never a stale oracle/_ref built from another checkout
    assert O.ref_lib() is not None, "oracle/_ref/libref_hsb_ops.so missing (no hsb_ops.cpp under %s)" % reference
    rng = np.random.default_rng(20260417)
    out = {}
    pi = np.fromfile(os.path.join(G, "fixture_prep_node_parent_idxs.i32"), np.int32)
    js = np.fromfile(os.path.join(G, "fixture_prep_node_js.i32"), np.int32)
    cases = {"fixture_shared": (pi, js, 6, True)}
    p2, j2 = synth.random_tree(97, seed=5)
    cases["random97_shared"] = (p2, j2, 5, True)
    cases["per_row"] = (None, None, 4, False)
    for name, (pi_, js_, B, shared) in cases.items():
        if shared:
            l, r, f = O.make_inverse_ptt_params(pi_, js_)
            n = (len(js_) + 1) // 2
            L, R, F = (np.broadcast_to(a, (B, len(a))).copy() for a in (l, r, f))
        else:
            n = 61
            trees = [O.make_inverse_ptt_params(*synth.random_tree(n, seed=100 + b)) for b in range(B)]
            L, R, F = (np.stack([t[i] for t in trees]) for i in range(3))
        y_logit = rng.normal(0, 2.5, (B, n - 1)).astype(np.float32)
        x = O.hsb(y_logit, L, R, F, impl="ref", threads=3)
        y, ladj = O.inv_hsb(x, L, R, F, impl="ref", threads=2)
        y_grad = rng.normal(size=(B, n - 1))
        ladj_grad = rng.normal(size=(B, 1)).astype(np.float32)
        bp = O.inv_hsb_grad(y_grad, ladj_grad, y, ladj, L, R, F, impl="ref", threads=2)
        for k, v in dict(left=L, right=R, leaf=F, y_logit=y_logit, x=x, y=y, ladj=ladj, y_grad=y_grad,
                         ladj_grad=ladj_grad, backprops=bp).items():
            out["%s__%s" % (name, k)] = v
    np.savez_compressed(os.path.join(G, "hsb_reference_vectors.npz"), **out)
    print("wrote", len(out), "arrays;", sorted(set(k.split("__")[0] for k in out)))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_hsb_vectors.py <polee checkout>")
    main(sys.argv[1])
