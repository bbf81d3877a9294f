#!/usr/bin/env python3
"""Generates tests/golden/reference_outputs.npz: what the unmodified reference computes on the inputs of
test_gpu_parity.py's comparisons with it (REF_CASES in fp64, FP32_CASES with its USE_FLOAT32 build).

Needs a GPU and oracle/_ref/libcuba_ref*.so, which build() compiles where the reference sources are present;
cases on the full ba_kitti_* graphs are stored only where their fixtures were extracted.  Per case: the chi2
trajectory (and the warm-up chi2 of the protocol cases), a seeded sample of the rows of q / t / Xw and of the
per-edge chi2 with the row indices, and the sum of absolute values of each whole array.

  python tests/golden/make_reference_golden.py [OUT.npz]"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle"), ROOT]
import __graft_entry__ as ge  # noqa: E402
import reference  # noqa: E402
from conftest import KERNELS, SUBGRAPHS, fixture_path, have_fixture, load_subgraph  # noqa: E402
from test_gpu_parity import FP32_CASES, REF_CASES, ref_problem  # noqa: E402

ROWS, EDGES = 32, 64


def put(out, key, name, a, k):
    a = np.asarray(a, dtype=np.float64)
    rows = np.sort(np.random.default_rng(len(a)).choice(len(a), min(len(a), k), replace=False)).astype(np.int32)
    out["%s__%s_rows" % (key, name)] = rows
    out["%s__%s" % (key, name)] = a[rows]
    out["%s__%s_abs_sum" % (key, name)] = np.array(np.abs(a).sum())


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "reference_outputs.npz")
    assert reference.available() and reference.available(fp32=True), "oracle/_ref/libcuba_ref*.so not built"
    pkg = ge.load_package()
    cache = {}

    def problems(name):
        if name not in cache:
            g = pkg.graphio.read_graph(fixture_path(name)) if name.startswith("ba_") else \
                load_subgraph(name) if name in SUBGRAPHS else pkg.synth.make_config(name)
            cache[name] = pkg.graphio.flatten(g)
        return cache[name]

    out = {}
    for name, kernel, how in REF_CASES:
        if name.startswith("ba_") and not have_fixture(name):
            continue
        key = "%s-%s-%s" % (name, kernel, how)
        rk = KERNELS[kernel]
        pr = ref_problem(pkg, problems(name), how)
        if how == "protocol":
            w = reference.run(pr, 1, *rk)
            out[key + "__warm_chi2"] = w["chi2"]
            pr = pr.copy(); pr.q, pr.t, pr.Xw = w["q"], w["t"], w["Xw"]
        r = reference.run(pr, 10, *rk, want_chisq=True)
        out[key + "__chi2"] = r["chi2"]
        for nme in ("q", "t", "Xw"):
            put(out, key, nme, r[nme], ROWS)
        put(out, key, "chisq", r["chisq"], EDGES)
        print(key, r["chi2"][-1], flush=True)
    for name, kernel in FP32_CASES:
        if name.startswith("ba_") and not have_fixture(name):
            continue
        key = "fp32-%s-%s" % (name, kernel)
        r = reference.run(problems(name), 10, *KERNELS[kernel], fp32=True)
        out[key + "__chi2"] = r["chi2"]
        for nme in ("t", "Xw"):
            put(out, key, nme, r[nme], ROWS)
        print(key, r["chi2"][-1], flush=True)
    np.savez_compressed(path, **out)
    print("wrote %s (%d bytes)" % (path, os.path.getsize(path)))


if __name__ == "__main__":
    main()
