"""Per-stage device times (L2 flushed) for one or more workloads.
usage: python tools/stage_bench.py <workload | ba_kitti_00> ..."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

pkg = ge.load_package()
args = sys.argv[1:]
NAMES = {1: "jh_landmark", 2: "jh_pose", 3: "schur", 4: "pcg", 5: "backsub+update+chi2", 6: "chi2"}
for workload in args or ["kitti00_shaped"]:
    if workload.startswith("ba_"):
        path = os.path.join(ROOT, "oracle", "_ref", "fixtures", workload + ".cubagraph")
        if not os.path.exists(path):
            print(workload, "fixture absent"); continue
        g = pkg.graphio.read_graph(path)
    else:
        g = pkg.synth.make_config(workload)
    prob = pkg.graphio.flatten(g)
    eng = pkg.Engine(device=0, use_fp32=("mixed" if os.environ.get("MIXED") else False))
    if os.environ.get("CUBA_DRY_SHARD"):
        r, w = os.environ["CUBA_DRY_SHARD"].split("/")
        eng.set_comm(int(r), int(w), b"\0" * 128)
    eng.initialize(prob)
    eng.linearize()
    lam = 1e-5 * eng.max_diagonal()
    eng.solve(lam)
    out = []
    for st in (1, 2, 3, 5, 6):
        out.append("%s %.1f us" % (NAMES[st], 1e3 * eng.bench_stage(st, reps=20, flush_l2=True, lam=lam)))
    print("%s: %s" % (workload, "; ".join(out)), flush=True)
    eng.close()
