#!/usr/bin/env python3
"""bench.py -- LM edges/s of the B200-native bundle-adjustment engine (metric of BASELINE.json).

One "step" = one pass of the hot path over one graph: `optimize(10)` (10 LM iterations, fp64 unless --fp32).

Workloads (BASELINE.json `configs`):
  N = 1 (default)  headline = C2, the reference's own fixture ba_kitti_00 (1 322 poses / 133 383 landmarks / 561 116 edges,
                   kernel NONE) under the reference's protocol: warm-up initialize()+optimize(1) written back, then the
                   timed initialize()+optimize(10) (samples/sample_ba_from_file.cpp:52-57,159-161).  The fixture travels in
                   oracle/_ref/fixtures (extracted by oracle/extract_fixtures.py); without it the seeded look-alike
                   `kitti00_shaped` is used and said so.  The line also carries `configs`: C1..C5, each measured here.
  N > 1            headline = C4, synth_stereo_10m (10 000 poses / 2 M landmarks / 10 M stereo edges, Huber), landmark-sharded,
                   reduced system row-distributed over the ranks (k_pcg5); kitti00_shaped rides along in `secondary`.

  value  : LM edge-iterations/s with every input already resident in HBM (state reset by a device copy,
           L2 flushed before each step), CUDA-event timed on the engine's stream, max over ranks.
  e2e    : the same metric through the reference-facing C ABI with HOST buffers: set_problem (H2D copies from pinned
           memory + structure build) + optimize(10) + get_state (D2H) per step -- the reference's own timed window.
  e2e_cpp: the same window through the drop-in C++ class cuba::CudaBundleAdjustment (samples/sample_ba_from_file --repeat):
           pointer-graph flattening (reference a1) included, wall clock inside the sample.
  roofline: the Jacobian+Hessian landmark-pass kernel (the HBM-dominant kernel), algorithmic bytes of
           SURVEY.md 8(d) / CUDA-event time per launch, against MEASURED_PEAKS.json.
  cpu_baseline: the CPU oracle (g2o-equivalent restatement, oracle/ba_oracle.c) on the same graph.

`--impl reference` times the UNMODIFIED reference (compiled for sm_100 into oracle/_ref/libcuba_ref.so by
oracle/build_ref.sh) through its own public API on the same workload and protocol -- the reference is a GPU library, so
its arm runs on the GPU; when the library is missing the arm falls back to the CPU oracle port.

Launch: python bench.py [--gpus N --steps K --warmup W] [--dump-outputs DIR]; for N>1 under torch.distributed.run.
Every workload, the headline and each of the configs, times K steps.  --dump-outputs writes what the last timed step of the
headline returned (chi2 / lambda / trials / pcg_iters per iteration, q, t, Xw) as DIR/<name>.npy; the inputs are the fixture or
a seeded graph, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import dataclasses
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

KERNELS = {"none": ((0, 0), (0.0, 0.0)), "huber": ((1, 1), (5.991 ** 0.5, 7.815 ** 0.5)), "tukey": ((2, 2), (4.0, 5.0))}
LM_ITERS = 10
README_K00 = [334210.0, 331822.8, 329700.4, 327743.4, 326123.2, 324876.6, 323698.5, 322572.7, 321410.3, 320086.4]   # reference README.md:141-150


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.rows = []

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def jh_bytes(sz, s=8):
    """SURVEY.md 8(d): algorithmic bytes of the Jacobian+Hessian stage.  Returns (landmark-pass kernel, whole stage)."""
    E2, E3, nhpl, Pall, Lall, P, L = sz["E2"], sz["E3"], sz["nhpl"], sz["Pall"], sz["Lall"], sz["numP"], sz["numL"]
    common = E2 * (3 * s + 8) + E3 * (4 * s + 8) + nhpl * 18 * s + Pall * 12 * s + Lall * 3 * s + L * 12 * s
    return common, common + P * 42 * s


def schur_bytes(sz, s=8):
    """SURVEY.md 8(d): B_S = nHpl 18 s + L 21 s + nblk 36 s + P 48 s"""
    return sz["nhpl"] * 18 * s + sz["numL"] * 21 * s + sz["nblk"] * 36 * s + sz["numP"] * 48 * s


def fixture_path(name):
    return os.path.join(ROOT, "oracle", "_ref", "fixtures", name + ".cubagraph")


def resolve_workload(name):
    """the reference's fixtures when they are on the box, their seeded look-alikes otherwise"""
    if name.startswith("ba_") and not os.path.exists(fixture_path(name)):
        return {"ba_kitti_00": "kitti00_shaped", "ba_kitti_07": "kitti07_shaped"}[name], "fixture %s absent -> seeded look-alike" % name
    return name, None


def load_graph(pkg, workload):
    return pkg.graphio.read_graph(fixture_path(workload)) if workload.startswith("ba_") else pkg.synth.make_config(workload)


def build_problem(pkg, workload):
    return pkg.graphio.flatten(load_graph(pkg, workload))


def golden_large():
    p = os.path.join(ROOT, "tests", "golden", "oracle_large.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def golden_small():
    p = os.path.join(ROOT, "tests", "golden", "oracle_trajectories.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def pin_problem(prob):
    """the e2e leg copies its inputs from PINNED host memory (bench contract): page-lock the flat problem once"""
    import torch

    def _pin(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy() if isinstance(a, np.ndarray) and a.size else a
    return dataclasses.replace(prob, **{f.name: _pin(getattr(prob, f.name)) for f in dataclasses.fields(prob)
                                        if f.name in ("q", "t", "cam", "Xw", "idx2", "meas2", "omega2", "idx3", "meas3", "omega3")})


class Runner:
    """one engine on this rank's GPU + the distributed plumbing of the timed loops"""

    def __init__(self, pkg, local, rank, world, fp32=False, mixed=False):
        import torch
        import torch.distributed as dist
        self.pkg, self.local, self.rank, self.world, self.fp32, self.mixed = pkg, local, rank, world, fp32, mixed
        self.torch, self.dist = torch, dist
        self.uid_fn = lambda: pkg.sharding.broadcast_unique_id(pkg.Engine, rank, world)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if self.world == 1:
            return ms
        t = self.torch.tensor([ms], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def engine(self, rk, **kw):
        eng = self.pkg.Engine(device=self.local, use_fp32=("mixed" if self.mixed else self.fp32), **kw)
        for et in (0, 1):
            eng.set_robust_kernels(rk[0][et], rk[1][et], et)
        if self.world > 1:
            eng.set_comm(self.rank, self.world, self.uid_fn())
        return eng

    def measure(self, prob, rk, steps, warmup, protocol_warmup=False, stages=True, clocks=None, keep_outputs=False):
        """returns a dict with value / e2e / roofline / stage times for one workload; with keep_outputs, also "outputs": what the
        last timed optimize(10) returned to its caller (per-iteration statistics and the final q / t / Xw)"""
        torch = self.torch
        pkg = self.pkg
        E = prob.nedges
        eng = self.engine(rk)
        warm_chi2 = None
        if protocol_warmup:
            # the reference's warm-up: initialize(); optimize(1); the result is written back into the graph
            eng.initialize(prob)
            w = eng.optimize(1)
            warm_chi2 = w[0]["chi2"]
            q, t, Xw = eng.state()
            prob = dataclasses.replace(prob, q=q, t=t, Xw=Xw)
        prob = pin_problem(prob)
        stream = torch.cuda.ExternalStream(eng.stream_ptr(), device=self.local)
        # ---------------- e2e with structure reuse (the product's default: an unchanged topology keeps every device structure)
        reuse_ms = []
        eng.initialize(prob)
        for i in range(2 + steps):
            self.barrier()
            a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
            a.record(stream)
            eng.initialize(prob)
            eng.optimize(LM_ITERS)
            eng.state()
            b.record(stream)
            self.barrier()
            if i >= 2:
                reuse_ms.append(self.max_over_ranks(a.elapsed_time(b)))
        reuses = eng.structure_reuses()
        # ---------------- e2e: host buffers -> set_problem (H2D + FULL structure build, like the reference) -> optimize -> get_state (D2H)
        eng.set_structure_reuse(False)
        e2e_ms, e2e_iters, h2d0, d2h0 = [], LM_ITERS, 0, 0
        for i in range(warmup + steps):
            if i == warmup:
                h2d0, d2h0 = pkg.transfer_bytes()
            self.barrier()
            a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
            a.record(stream)
            eng.initialize(prob)
            stats = eng.optimize(LM_ITERS)
            q, t, Xw = eng.state()
            b.record(stream)
            self.barrier()
            if i >= warmup:
                e2e_ms.append(self.max_over_ranks(a.elapsed_time(b))); e2e_iters = len(stats)
        h2d1, d2h1 = pkg.transfer_bytes()
        prof = eng.time_profile()     # buckets of exactly one e2e step (set_problem resets them)
        e2e_t = float(np.mean(e2e_ms)) * 1e-3
        sizes = eng.sizes
        # ---------------- value: inputs resident in HBM, L2 flushed, device-timed optimize(10)
        if clocks is not None:
            clocks.start()
        dev_ms, iters_done, launches0, pcg_total, pcg_ms0 = [], LM_ITERS, 0, 0, 0.0
        for i in range(warmup + steps):
            if i == warmup:
                launches0 = eng.launch_count()
                pcg_ms0 = 1e3 * eng.time_profile()["6: Numerical Decomposition"]
            eng.reset_state(); eng.flush_l2()
            self.barrier()
            a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
            a.record(stream)
            stats = eng.optimize(LM_ITERS)
            b.record(stream)
            self.barrier()
            if i >= warmup:
                dev_ms.append(self.max_over_ranks(a.elapsed_time(b))); iters_done = len(stats)
                pcg_total = sum(s["pcg_iters"] for s in stats)
        launches = eng.launch_count() - launches0
        outputs = None
        if keep_outputs:
            q, t, Xw = eng.state()
            outputs = {"chi2": [s["chi2"] for s in stats], "lambda": [s["lambda_"] for s in stats], "trials": [s["trials"] for s in stats],
                       "pcg_iters": [s["pcg_iters"] for s in stats], "q": q, "t": t, "Xw": Xw}
        pcg_ms = (1e3 * eng.time_profile()["6: Numerical Decomposition"] - pcg_ms0) / max(steps, 1)
        if clocks is not None:
            clocks.stop_flag.set(); clocks.join(timeout=3)
        ms_per_step = float(np.mean(dev_ms))
        out = {"E": E, "sizes": sizes, "value": E * iters_done / (ms_per_step * 1e-3), "ms_per_step": ms_per_step, "iters": iters_done,
               "chi2": [s["chi2"] for s in stats], "trials": [s["trials"] for s in stats], "final_chi2": stats[-1]["chi2"], "warmup_chi2": warm_chi2,
               "pcg_iterations_per_step": pcg_total, "pcg_ms_per_step": pcg_ms, "pcg_us_per_iteration": 1e3 * pcg_ms / max(pcg_total, 1),
               "launches": launches,
               "e2e": {"value": E * e2e_iters / e2e_t, "unit": "edge-iterations/s", "ms_per_step": 1e3 * e2e_t,
                       "h2d_bytes_per_step": (h2d1 - h2d0) // max(steps, 1), "d2h_bytes_per_step": (d2h1 - d2h0) // max(steps, 1),
                       "window": "set_problem(H2D from pinned host buffers + full structure build, structure reuse switched OFF) + optimize(10) + get_state(D2H) == reference's initialize()+optimize(10)"},
               "e2e_reuse": {"value": E * e2e_iters / (float(np.mean(reuse_ms)) * 1e-3), "unit": "edge-iterations/s", "ms_per_step": float(np.mean(reuse_ms)), "structure_reuses": reuses,
                             "window": "the same window with the engine's default structure reuse: the topology is unchanged between calls, so set_problem only uploads values (SURVEY 8 f-2)"},
               "profile_ms_e2e_step": {k: round(1e3 * v, 4) for k, v in prof.items()}, "prob": prob, "outputs": outputs}
        # ---------------- roofline of the J+H landmark-pass kernel + per-stage device times (L2 flushed between reps)
        if stages:
            eng.reset_state(); eng.linearize()
            lam = 1e-5 * eng.max_diagonal()
            stage_ms = {}
            for label, st in (("jh_landmark_pass", 1), ("jh_pose_pass", 2), ("schur", 3), ("pcg_solve", 4), ("backsub_update_chi2", 5), ("chi2_only", 6)):
                stage_ms[label] = eng.bench_stage(st, reps=20 if E < 2000000 else 5, flush_l2=True, lam=lam)
            s = 4 if self.fp32 else 8
            b_kernel, b_stage = jh_bytes(sizes, s)          # per-rank bytes: each rank streams its shard of the edges
            if self.mixed:
                b_kernel -= sizes["nhpl"] * (144 - 80); b_stage -= sizes["nhpl"] * (144 - 80)   # 80-byte fp32 Hpl blocks
            b_kernel /= self.world; b_stage /= self.world
            peak, peak_src = measured_peak()
            ach = b_kernel / (stage_ms["jh_landmark_pass"] * 1e-3) / 1e9
            out["stage_ms"] = stage_ms
            out["roofline"] = {"bound": "hbm", "kernel": ("k_linearize_landmark<float>" if self.fp32 else "k_linearize_landmark4"), "achieved": ach,
                               "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src, "algorithmic_bytes": b_kernel,
                               "ms_per_launch": stage_ms["jh_landmark_pass"],
                               "stage_frac_jh_both_kernels": b_stage / ((stage_ms["jh_landmark_pass"] + stage_ms["jh_pose_pass"]) * 1e-3) / 1e9 / peak,
                               "schur_frac": schur_bytes(sizes, s) / self.world / (stage_ms["schur"] * 1e-3) / 1e9 / peak}
        eng.close()
        return out


def cpu_reference_chi2(prob, rk):
    """live CPU oracle run (rank 0): (final chi2, edge-iterations/s, seconds)"""
    oracle = ge.load_oracle()
    o = oracle.Oracle(prob, rk[0], rk[1])
    t0 = time.perf_counter(); chi, lam_o, tr = o.optimize(LM_ITERS); dt = time.perf_counter() - t0
    return chi, prob.nedges * len(chi) / dt, dt


DUMP_BYTES = 64 << 20


def dump_outputs(outputs, out_dir):
    """--dump-outputs: one <name>.npy per output of the last timed step, float32 / float64, so that two builds can be compared
    output for output.  Beyond 64 MB in all, Xw keeps a fixed seeded sample of its rows, whose indices go to Xw_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {}
    for name, v in outputs.items():
        a = np.asarray(v)
        arrays[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        Xw = arrays["Xw"]
        k = (DUMP_BYTES - (total - Xw.nbytes)) // (Xw.itemsize * Xw.shape[1] + 8)
        rows = np.sort(np.random.default_rng(0).choice(len(Xw), k, replace=False))
        arrays["Xw"], arrays["Xw_rows"] = Xw[rows], rows.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_e2e_cpp(pkg, workload, graph, robust, steps, warmup, reuse=True):
    """initialize()+optimize(10) through cuba::CudaBundleAdjustment: the sample binary times the window itself (--repeat)"""
    tmp = tempfile.mkdtemp(prefix="cuba_bench_")
    exe = os.path.join(tmp, "sample_ba_from_file")
    libdir = os.path.dirname(pkg.library_path())
    try:
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-DCUBA_FORCE_EIGEN_COMPAT", "-I", os.path.join(ROOT, "include"),
                               os.path.join(ROOT, "samples", "sample_ba_from_file.cpp"), "-L", libdir, "-lcuba_b200", "-Wl,-rpath," + libdir, "-o", exe])
        path = fixture_path(workload)
        if not workload.startswith("ba_"):
            path = os.path.join(tmp, workload + ".cubagraph")
            pkg.graphio.write_graph(path, graph)
        env = dict(os.environ)
        if not reuse:
            env["CUBA_NO_STRUCTURE_REUSE"] = "1"
        res = subprocess.run([exe, path, "--json", "--repeat", str(warmup + steps)] + (["--huber"] if robust == "huber" else []),
                             capture_output=True, text=True, timeout=900, env=env)
        if res.returncode != 0:
            return {"error": res.stderr[-300:]}
        r = json.loads(res.stdout)
        secs = r["seconds_all"][warmup:]
        sec = float(np.mean(secs))
        return {"value": r["nedges"] * len(r["chi2"]) / sec, "unit": "edge-iterations/s", "ms_per_step": 1e3 * sec, "final_chi2": r["chi2"][-1],
                "profile_ms": {k: round(1e3 * v, 4) for k, v in r["profile"].items()},
                "structure_reuse": bool(reuse),
                "window": "cuba::CudaBundleAdjustment::initialize() + optimize(10) (pointer graph -> flat arrays -> C ABI), wall clock inside samples/sample_ba_from_file --repeat"}
    except Exception as ex:   # the C++ leg must never take the bench line down
        return {"error": str(ex)[-300:]}


def run_reference(args, pkg, rk, rank):
    """--impl reference: the compiled reference (GPU build) through its own API; CPU oracle port if absent."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reference
    import torch
    prob = build_problem(pkg, args.workload)
    E = prob.nedges
    use_ref = reference.available(args.fp32) and torch.cuda.is_available()
    times, iters, chi2 = [], LM_ITERS, []
    kind, sample = "reference", ""
    nwarm, nsteps = args.warmup, args.steps
    if E > 2000000:
        # multi-million-edge workloads: a bounded sample of runs so that the arm ends within a few minutes (one run is several seconds)
        nwarm, nsteps = min(nwarm, 1), min(nsteps, 2)
    if use_ref:
        if args.protocol_warmup:
            w = reference.run(prob, 1, rk[0], rk[1], fp32=args.fp32)      # the reference's own warm-up, written back
            if w is not None:
                prob = dataclasses.replace(prob, q=w["q"], t=w["t"], Xw=w["Xw"])
        for i in range(nwarm + nsteps):
            r = reference.run(prob, LM_ITERS, rk[0], rk[1], warmup=0, fp32=args.fp32)
            if r is None:
                use_ref = False
                break
            if i >= nwarm:
                times.append(r["seconds"]); iters = len(r["chi2"]); chi2 = [float(v) for v in r["chi2"]]
        sample = "unmodified reference compiled for sm_100 (oracle/_ref/libcuba_ref.so), initialize()+optimize(10) on the full graph, " \
                 "host buffers, %d timed runs after %d warm-up; runs on the GPU because the reference has no CPU path (its CPU comparator g2o is not in the image)" % (nsteps, nwarm)
    if not use_ref or not times:
        kind = "port"
        oracle = ge.load_oracle()
        for i in range(min(args.warmup, 1) + min(args.steps, 2)):
            o = oracle.Oracle(prob, rk[0], rk[1])
            t0 = time.perf_counter(); chi, lam, tr = o.optimize(LM_ITERS); dt = time.perf_counter() - t0
            if i >= min(args.warmup, 1):
                times.append(dt); iters = len(chi); chi2 = [float(v) for v in chi]
        sample = "CPU oracle port (oracle/ba_oracle.c), optimize(10) on the full graph"
    sec = float(np.mean(times))
    val = E * iters / sec
    cores = 1 if kind == "port" else 0
    line = {"impl": "reference", "metric": "LM edges/sec (10 iters)", "value": val, "unit": "edge-iterations/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32" if args.fp32 else "f64", "data": args.data,
            "config": {"workload": args.workload, "robust_kernel": args.robust, "lm_iterations": LM_ITERS, "edges": E,
                       "protocol": "warm-up optimize(1) written back, then initialize()+optimize(10)" if args.protocol_warmup else "initialize()+optimize(10) from the generated estimate"},
            "chi2_per_iteration": chi2,
            "cpu_baseline": {"value": val, "unit": "edge-iterations/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": val, "unit": "edge-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if rank == 0:
        print(json.dumps(line), flush=True)


def config_entry(name, workload, robust, fp32, m, oracle_chi2, oracle_kind):
    e = {"config": name, "workload": workload, "robust_kernel": robust, "dtype": "f32" if fp32 is True else ("f64 (Hpl stored in f32)" if fp32 == "mixed" else "f64"), "edges": m["E"],
         "value": m["value"], "ms_per_step": m["ms_per_step"], "e2e": m["e2e"]["value"], "e2e_ms_per_step": m["e2e"]["ms_per_step"],
         "roofline_frac": m["roofline"]["frac"] if "roofline" in m else None, "jh_landmark_pass_us": 1e3 * m["stage_ms"]["jh_landmark_pass"] if "stage_ms" in m else None,
         "schur_us": 1e3 * m["stage_ms"]["schur"] if "stage_ms" in m else None,
         "stage_frac_jh_both_kernels": m["roofline"]["stage_frac_jh_both_kernels"] if "roofline" in m else None,
         "schur_frac": m["roofline"]["schur_frac"] if "roofline" in m else None,
         "pcg_iterations_per_step": m["pcg_iterations_per_step"], "pcg_ms_per_step": m["pcg_ms_per_step"],
         "final_chi2": m["final_chi2"], "chi2_rel_diff_vs_oracle": None, "oracle": oracle_kind}
    if oracle_chi2 is not None and len(oracle_chi2) == len(m["chi2"]):
        e["chi2_rel_diff_vs_oracle"] = float(np.abs(np.array(m["chi2"]) - np.array(oracle_chi2)).max() / np.abs(oracle_chi2).max())
    return e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, help="default: ba_kitti_00 on one GPU, synth_stereo_10m on several")
    ap.add_argument("--robust", default=None, choices=list(KERNELS))
    ap.add_argument("--fp32", action="store_true")
    ap.add_argument("--mixed", action="store_true", help="fp64 engine with the Hpl blocks stored in fp32 (SURVEY 8 f-4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the C1..C5 array (and, on several GPUs, the secondary workload)")
    ap.add_argument("--no-cpp", action="store_true")
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (chi2, lambda, trials, pcg_iters per iteration; q, t, Xw) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps this engine's outputs: use it with --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    explicit = args.workload is not None
    if args.workload is None:
        args.workload = "ba_kitti_00" if world == 1 and args.gpus == 1 else "synth_stereo_10m"
    args.workload, note = resolve_workload(args.workload)
    if args.robust is None:
        args.robust = "huber" if args.workload.startswith("synth_") else "none"
    args.protocol_warmup = args.workload.startswith("ba_")
    args.data = "reference fixture (samples/ba_input.7z)" if args.workload.startswith("ba_") else "synthetic"
    rk = KERNELS[args.robust]
    pkg = ge.load_package()

    if args.impl == "reference":
        if rank != 0:
            return 0      # rank 0 alone runs and prints the reference arm
        big = args.workload.startswith("synth_") and args.workload != "synth_small"
        if big and not args.child:
            # the reference was written for KITTI-sized graphs: on the multi-million-edge workloads it runs in a child process under a
            # time limit, so that a failure or a run of many minutes yields the documented "unavailable" line instead of a hang
            cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--child", "--gpus", str(args.gpus), "--steps", str(args.steps),
                   "--warmup", str(args.warmup), "--workload", args.workload, "--robust", args.robust] + (["--fp32"] if args.fp32 else [])
            env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT")}
            try:
                res = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=env)
                lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
                if res.returncode == 0 and lines:
                    print(lines[-1], flush=True)
                else:
                    print(json.dumps({"impl": "reference", "unavailable": "the reference GPU build failed on %s (exit code %d): %s" % (args.workload, res.returncode, (res.stderr or "")[-160:].replace("\n", " "))}), flush=True)
            except subprocess.TimeoutExpired:
                print(json.dumps({"impl": "reference", "unavailable": "the reference GPU build did not finish initialize()+optimize(10) runs on %s within 420 s" % args.workload}), flush=True)
            return 0
        run_reference(args, pkg, rk, rank)
        return 0

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    run = Runner(pkg, local, rank, world, fp32=args.fp32, mixed=args.mixed)

    graph = load_graph(pkg, args.workload)
    prob0 = pkg.graphio.flatten(graph)
    clocks = ClockSampler(local)
    m = run.measure(prob0, rk, args.steps, args.warmup, protocol_warmup=args.protocol_warmup, clocks=clocks, keep_outputs=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(m["outputs"], args.dump_outputs)
    E, sizes = m["E"], m["sizes"]
    tpath = os.path.join(ROOT, "profiles", "jh_traffic.json")
    if os.path.exists(tpath) and world == 1:
        try:
            m["roofline"]["traffic"] = json.load(open(tpath)).get(args.workload)
        except Exception:
            pass

    # ---------------- chi2 against the oracle: live on the KITTI-sized graphs, committed goldens on the multi-million-edge ones
    gl, gs = golden_large(), golden_small()
    chi_oracle, oracle_kind, cpu = None, None, None
    if rank == 0:
        if E <= 1000000 and world == 1 and not args.no_cpu_baseline and not args.fp32:
            chi_o, cpu_val, dt = cpu_reference_chi2(m["prob"], rk)
            chi_oracle, oracle_kind = chi_o, "live (oracle/ba_oracle.c on this box)"
            cpu = {"value": cpu_val, "unit": "edge-iterations/s", "cores": 1, "kind": "port",
                   "sample": "oracle/ba_oracle.c (g2o-equivalent: Schur + sparse block Cholesky + LM), one optimize(10) on the full %s graph, %.1f s; "
                             "host has %d cores, the port is single-threaded like g2o's default" % (args.workload, dt, os.cpu_count()),
                   "final_chi2": float(chi_o[-1]), "chi2_rel_diff_vs_gpu": float(abs(chi_o[-1] - m["final_chi2"]) / chi_o[-1])}
        else:
            key = "%s_%s" % (args.workload, args.robust)
            if key in gl and not args.fp32:
                chi_oracle, oracle_kind = gl[key]["chi2"], "golden (tests/golden/oracle_large.json, CPU oracle run offline, %.0f s)" % gl[key].get("oracle_seconds", 0)
            elif key in gs and not args.fp32:
                chi_oracle, oracle_kind = gs[key]["chi2"], "golden (tests/golden/oracle_trajectories.json)"
    chi_rel = None
    if chi_oracle is not None and len(chi_oracle) == len(m["chi2"]):
        chi_rel = float(np.abs(np.array(m["chi2"]) - np.array(chi_oracle)).max() / np.abs(chi_oracle).max())

    line = {"metric": "LM edges/sec (10 iters)", "value": m["value"], "unit": "edge-iterations/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32" if args.fp32 else "f64", "data": args.data,
            "config": {"workload": args.workload, "poses": sizes["Pall"], "landmarks": sizes["Lall"], "edges": E, "robust_kernel": args.robust,
                       "lm_iterations": m["iters"], "l2": "flushed between timed steps (320 MB fill)",
                       "parallelism": "landmark-sharded x%d%s" % (world, ", reduced system row-distributed over the ranks (k_pcg5, NVLink peer boards)" if world > 1 and sizes["numP"] >= 2048 else ""),
                       "protocol": "reference: warm-up optimize(1) written back, then initialize()+optimize(10)" if args.protocol_warmup else "initialize()+optimize(10) from the generated estimate",
                       "pcg_iterations_per_step": m["pcg_iterations_per_step"], "final_chi2": m["final_chi2"]},
            "e2e": m["e2e"], "e2e_reuse": m["e2e_reuse"], "gpu_launches": m["launches"], "clocks": clocks.summary(), "roofline": m["roofline"], "stage_ms": m["stage_ms"],
            "profile_ms_e2e_step": m["profile_ms_e2e_step"],
            "pcg": {"iterations_per_step": m["pcg_iterations_per_step"], "ms_per_step": m["pcg_ms_per_step"], "us_per_iteration": m["pcg_us_per_iteration"]},
            "chi2_per_iteration": m["chi2"], "chi2_rel_diff_vs_oracle": chi_rel, "oracle": oracle_kind}
    if note:
        line["config"]["note"] = note
    if args.workload == "ba_kitti_00" and args.robust == "none" and not args.fp32:
        line["readme_chi2_table"] = {"reference_README_md_141_150": README_K00, "this_run": [round(c, 1) for c in m["chi2"]],
                                     "max_abs_diff": float(np.abs(np.array(m["chi2"]) - np.array(README_K00)).max()) if len(m["chi2"]) == 10 else None}
    if cpu:
        line["cpu_baseline"] = cpu

    # ---------------- e2e through the drop-in C++ class (one GPU)
    if world == 1 and rank == 0 and not args.no_cpp and not args.fp32:
        line["e2e_cpp"] = run_e2e_cpp(pkg, args.workload, graph, args.robust, args.steps, args.warmup, reuse=False)
        line["e2e_cpp_reuse"] = run_e2e_cpp(pkg, args.workload, graph, args.robust, args.steps, args.warmup, reuse=True)

    # ---------------- the other BASELINE configs, each measured here (one GPU) / the KITTI-sized graph beside the 10 M-edge one (several GPUs)
    if not args.no_configs and not explicit and not args.fp32:
        if world == 1:
            configs = [config_entry("C2", args.workload, args.robust, False, m, chi_oracle, oracle_kind)]
            # (config, workload, robust kernel, precision, warm-up steps); every config times --steps steps
            plan = [("C1", "ba_kitti_07", "none", False, 3), ("C1", "ba_kitti_07", "huber", False, 3), ("C2", "ba_kitti_00", "huber", False, 3),
                    ("C5", "ba_kitti_00", "none", True, 3), ("C5-mixed", "ba_kitti_00", "none", "mixed", 3),
                    ("C3", "synth_mono_5m", "huber", False, 1), ("C4", "synth_stereo_10m", "huber", False, 1)]
            for name, wl, rb, f32, wu in plan:
                wl, _ = resolve_workload(wl)
                try:
                    p = build_problem(pkg, wl)
                    r2 = Runner(pkg, local, rank, world, fp32=(f32 is True), mixed=(f32 == "mixed"))
                    mm = r2.measure(p, KERNELS[rb], args.steps, wu, protocol_warmup=wl.startswith("ba_"))
                    oc, ok_ = None, None
                    if not f32:
                        if wl.startswith("ba_"):
                            key = "%s_%s" % (wl, rb)
                            if key in gs:
                                oc, ok_ = gs[key]["chi2"], "golden (tests/golden/oracle_trajectories.json, reference protocol)"
                        elif "%s_%s" % (wl, rb) in gl:
                            oc, ok_ = gl["%s_%s" % (wl, rb)]["chi2"], "golden (tests/golden/oracle_large.json)"
                        elif mm["E"] <= 1000000:
                            oc, ok_ = cpu_reference_chi2(mm["prob"], KERNELS[rb])[0], "live"
                    ent = config_entry(name, wl, rb, f32, mm, oc, ok_)
                    if f32:
                        # C5: chi2 tolerance vs fp64 = deviation of the fp32 trajectory from the fp64 run of the same protocol
                        ent["chi2_rel_diff_vs_fp64"] = float(np.abs(np.array(mm["chi2"]) - np.array(m["chi2"])).max() / np.abs(m["chi2"]).max()) if len(mm["chi2"]) == len(m["chi2"]) else None
                    ent["steps"], ent["warmup"] = args.steps, wu
                    configs.append(ent)
                    del mm, p
                except Exception as ex:
                    configs.append({"config": name, "workload": wl, "robust_kernel": rb, "error": str(ex)[-200:]})
            line["configs"] = configs
            # the N > 1 headline workload measured on ONE GPU in this same run: the base of the strong-scaling curve
            c4 = [c for c in configs if c.get("config") == "C4" and "value" in c]
            if c4:
                line["scaling_base"] = {"workload": c4[0]["workload"], "n_gpus": 1, "value": c4[0]["value"], "ms_per_step": c4[0]["ms_per_step"],
                                        "note": "bench.py --gpus N>1 runs this workload; divide its value by N x this value for the scaling efficiency"}
        else:
            try:
                p = build_problem(pkg, "kitti00_shaped")
                mm = run.measure(p, KERNELS["none"], args.steps, 3, stages=False)
                oc = gl.get("kitti00_shaped_none", {}).get("chi2")
                line["secondary"] = config_entry("kitti00_shaped (strong scaling of a latency-bound graph)", "kitti00_shaped", "none", False, mm, oc, "golden (tests/golden/oracle_large.json)" if oc else None)
            except Exception as ex:
                line["secondary"] = {"error": str(ex)[-200:]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
