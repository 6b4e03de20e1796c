#!/usr/bin/env python3
"""Convert the reference's two HDF5 test fixtures into flat little-endian binaries.

Run once on a checkout of the original Polee; the outputs are committed under tests/golden/
so that the tests need none.

    python tests/golden/make_fixtures.py <polee checkout>

Inputs (reference test data, SURVEY.md section 4 / 8c):
  test/dataset/mBr_M_6w_1.likelihood-matrix.h5   written by rnaseq_sample.jl:505-519
  test/dataset/mBr_M_6w_1.prep.h5                written by likelihood-approximation.jl:61-87

No HDF5 library exists in this image; polee_b200/h5min.py reads exactly the HDF5 features
those two files use (superblock v0, v1 object headers, compact link messages or a single
fractal-heap direct block, contiguous / chunked+deflate layouts).
"""
import hashlib
import json
import os
import struct
import sys
import zlib

import numpy as np

OUT = os.path.dirname(os.path.abspath(__file__))


sys.path.insert(0, os.path.dirname(os.path.dirname(OUT)))
from polee_b200.h5min import read_dataset, root_links  # noqa: E402  (the reader lives in the package: SURVEY 8f-3)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main(reference):
    ref = os.path.join(reference, "test", "dataset")
    manifest = {}

    def dump(name, arr):
        arr = np.ascontiguousarray(arr)
        path = os.path.join(OUT, name)
        arr.tofile(path)
        manifest[name] = {"dtype": str(arr.dtype), "count": int(arr.size), "sha256": sha(arr)}

    lm = open(os.path.join(ref, "mBr_M_6w_1.likelihood-matrix.h5"), "rb").read()
    links = root_links(lm)
    m = int(read_dataset(lm, links["m"])[0])
    n = int(read_dataset(lm, links["n"])[0])
    colptr = read_dataset(lm, links["colptr"])
    rowval = read_dataset(lm, links["rowval"])
    nzval = read_dataset(lm, links["nzval"])
    efflens = read_dataset(lm, links["effective_lengths"])
    assert colptr.dtype == np.uint32 and rowval.dtype == np.uint32
    assert nzval.dtype == np.float32 and efflens.dtype == np.float32
    assert len(colptr) == n + 1 and colptr[0] == 1 and colptr[-1] == len(rowval) + 1
    assert len(nzval) == len(rowval) and rowval.min() == 1 and rowval.max() == m
    dump("fixture_colptr.u32", colptr)
    dump("fixture_rowval.u32", rowval)
    dump("fixture_nzval.f32", nzval)
    dump("fixture_efflens.f32", efflens)

    pp = open(os.path.join(ref, "mBr_M_6w_1.prep.h5"), "rb").read()
    links = root_links(pp)
    assert int(read_dataset(pp, links["m"])[0]) == m
    assert int(read_dataset(pp, links["n"])[0]) == n
    eff2 = read_dataset(pp, links["effective_lengths"])
    assert eff2.tobytes() == efflens.tobytes()
    for key, dt in (("mu", np.float32), ("omega", np.float32), ("alpha", np.float32),
                    ("node_parent_idxs", np.int32), ("node_js", np.int32)):
        a = read_dataset(pp, links[key])
        assert a.dtype == dt, (key, a.dtype)
        dump("fixture_prep_%s.%s" % (key, "f32" if dt == np.float32 else "i32"), a)
    manifest["_meta"] = {"m": m, "n": n, "nnz": int(len(rowval)),
                         "source": ["test/dataset/mBr_M_6w_1.likelihood-matrix.h5",
                                    "test/dataset/mBr_M_6w_1.prep.h5"]}
    with open(os.path.join(OUT, "fixture_manifest.json"), "w") as fh:
        json.dump(manifest, fh, indent=1, sort_keys=True)
    print(json.dumps(manifest["_meta"]))
    for k, v in sorted(manifest.items()):
        if k != "_meta":
            print(k, v["count"], v["sha256"][:16])


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tests/golden/make_fixtures.py <polee checkout>")
    sys.exit(main(sys.argv[1]))
