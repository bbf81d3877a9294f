"""J+H landmark-pass variants: device time per launch (L2 flushed) on one workload.
usage: python tools/jh_variants.py [--variants 0,4] <workload | ba_kitti_00 | ba_kitti_07> ..."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

pkg = ge.load_package()
args = sys.argv[1:]
variants = (0, 4)
if args and args[0] == "--variants":
    variants = tuple(int(v) for v in args[1].split(","))
    args = args[2:]
for workload in args or ["kitti00_shaped"]:
    if workload.startswith("ba_"):
        path = os.path.join(ROOT, "oracle", "_ref", "fixtures", workload + ".cubagraph")
        if not os.path.exists(path):
            print(workload, "fixture absent"); continue
        g = pkg.graphio.read_graph(path)
    else:
        g = pkg.synth.make_config(workload)
    prob = pkg.graphio.flatten(g)
    for v in variants:
        eng = pkg.Engine(device=0, jh_variant=v)
        eng.initialize(prob)
        chi = eng.linearize()
        ms1 = eng.bench_stage(1, reps=30, flush_l2=True)
        ms1w = eng.bench_stage(1, reps=30, flush_l2=False)
        print("%s jh_variant %d: landmark pass %.1f us (L2 flushed) %.1f us (warm); chi2 %.9g" % (workload, v, 1e3 * ms1, 1e3 * ms1w, chi), flush=True)
        eng.close()
