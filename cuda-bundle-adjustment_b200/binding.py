"""ctypes binding of libcuba_b200.so (include/cuba_b200.h).  Mirrors the reference's operator interface
for the hot path: initialize()/optimize(n)/batchStatistics()/timeProfile()/chiSquared()
(reference include/cuda_bundle_adjustment.h:34-125) on a flat problem."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROBUST_NONE, ROBUST_HUBER, ROBUST_TUKEY = 0, 1, 2
EDGE_MONOCULAR, EDGE_STEREO = 0, 1
# reference src/cuda_bundle_adjustment.cpp:547-557
PROFILE_ITEMS = ("0: Initialize Optimizer", "1: Build Structure", "2: Compute Error", "3: Build System",
                 "4: Schur Complement", "5: Symbolic Decomposition", "6: Numerical Decomposition", "7: Update Solution")


class CubaError(RuntimeError):
    pass


def library_path():
    return os.path.join(HERE, "libcuba_b200.so")


class _Config(C.Structure):
    _fields_ = [("device", C.c_int), ("use_fp32", C.c_int), ("pcg_max_iters", C.c_int), ("pcg_tol", C.c_double),
                ("deterministic", C.c_int), ("reserved", C.c_int * 7)]


class _Problem(C.Structure):
    _fields_ = [("Pall", C.c_int32), ("numP", C.c_int32), ("Lall", C.c_int32), ("numL", C.c_int32),
                ("q", C.c_void_p), ("t", C.c_void_p), ("cam", C.c_void_p), ("Xw", C.c_void_p),
                ("E2", C.c_int32), ("idx2", C.c_void_p), ("meas2", C.c_void_p), ("omega2", C.c_void_p),
                ("E3", C.c_int32), ("idx3", C.c_void_p), ("meas3", C.c_void_p), ("omega3", C.c_void_p)]


class _IterStat(C.Structure):
    _fields_ = [("iteration", C.c_int32), ("trials", C.c_int32), ("chi2", C.c_double), ("lambda_", C.c_double),
                ("pcg_iters", C.c_int32), ("pcg_failed", C.c_int32)]


class _Sizes(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("Pall", "numP", "Lall", "numL", "E2", "E3", "nhpl", "nblk", "nmul", "nblk_full")]


_lib = None

_SYMBOLS = [
    "cuba_last_error", "cuba_version", "cuba_engine_create", "cuba_engine_destroy", "cuba_engine_set_robust_kernel",
    "cuba_comm_unique_id", "cuba_engine_set_comm", "cuba_engine_set_problem", "cuba_engine_set_structure_reuse", "cuba_engine_get_structure_reuses", "cuba_engine_set_state", "cuba_engine_get_sizes", "cuba_engine_reset_state", "cuba_engine_get_stream", "cuba_engine_flush_l2",
    "cuba_engine_optimize", "cuba_engine_get_state", "cuba_engine_get_chi2", "cuba_engine_get_profile",
    "cuba_engine_get_launch_count", "cuba_get_transfer_bytes", "cuba_stage_linearize", "cuba_stage_max_diagonal", "cuba_stage_solve", "cuba_stage_update",
    "cuba_stage_commit", "cuba_stage_chi2", "cuba_debug_get_hpl_structure", "cuba_debug_get_hsc_structure",
    "cuba_debug_get_system", "cuba_debug_get_schur", "cuba_debug_get_delta", "cuba_debug_build_structure_host", "cuba_debug_pcg_partition", "cuba_debug_pcg5_plan", "cuba_debug_dropin_problem", "cuba_bench_stage",
]


def exported_symbols():
    return list(_SYMBOLS)


def load_library():
    """Loads the in-tree libcuba_b200.so; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise CubaError("%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)" % path)
    L = C.CDLL(path)
    L.cuba_last_error.restype = C.c_char_p
    vp, i, d = C.c_void_p, C.c_int, C.c_double
    sig = {
        "cuba_engine_create": [C.POINTER(_Config), C.POINTER(vp)],
        "cuba_engine_destroy": [vp],
        "cuba_engine_set_robust_kernel": [vp, i, i, d],
        "cuba_comm_unique_id": [vp],
        "cuba_engine_set_comm": [vp, i, i, vp],
        "cuba_engine_set_problem": [vp, C.POINTER(_Problem)],
        "cuba_engine_set_structure_reuse": [vp, i],
        "cuba_engine_get_structure_reuses": [vp, C.POINTER(C.c_longlong)],
        "cuba_engine_set_state": [vp, vp, vp, vp],
        "cuba_engine_get_sizes": [vp, C.POINTER(_Sizes)],
        "cuba_engine_reset_state": [vp],
        "cuba_engine_get_stream": [vp, C.POINTER(vp)],
        "cuba_engine_flush_l2": [vp],
        "cuba_engine_optimize": [vp, i, vp, C.POINTER(i)],
        "cuba_engine_get_state": [vp, vp, vp, vp],
        "cuba_engine_get_chi2": [vp, vp],
        "cuba_engine_get_profile": [vp, vp],
        "cuba_engine_get_launch_count": [vp, C.POINTER(C.c_longlong)],
        "cuba_get_transfer_bytes": [C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)],
        "cuba_stage_linearize": [vp, C.POINTER(d)],
        "cuba_stage_max_diagonal": [vp, C.POINTER(d)],
        "cuba_stage_solve": [vp, d, C.POINTER(i), C.POINTER(i)],
        "cuba_stage_update": [vp, d, C.POINTER(d), C.POINTER(d)],
        "cuba_stage_commit": [vp, i],
        "cuba_stage_chi2": [vp, C.POINTER(d)],
        "cuba_debug_get_hpl_structure": [vp, vp, vp, vp],
        "cuba_debug_get_hsc_structure": [vp, vp, vp],
        "cuba_debug_get_system": [vp, vp, vp, vp, vp, vp],
        "cuba_debug_get_schur": [vp, vp, vp, vp],
        "cuba_debug_get_delta": [vp, vp, vp],
        "cuba_debug_build_structure_host": [C.POINTER(_Problem), i, i, C.POINTER(_Sizes), vp, vp, vp, vp, vp, vp, vp, vp],
        "cuba_debug_pcg_partition": [C.POINTER(_Problem), i, i, vp],
        "cuba_debug_pcg5_plan": [C.POINTER(_Problem), i, i, i, vp],
        "cuba_debug_dropin_problem": [vp, C.POINTER(_Problem)],
        "cuba_bench_stage": [vp, i, i, i, d, C.POINTER(d)],
    }
    for name, args in sig.items():
        fn = getattr(L, name)
        fn.argtypes = args
        fn.restype = C.c_int
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise CubaError("cuba error %d: %s" % (rc, load_library().cuba_last_error().decode()))


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _problem_struct(prob):
    keep = [np.ascontiguousarray(prob.q, dtype=np.float64), np.ascontiguousarray(prob.t, dtype=np.float64),
            np.ascontiguousarray(prob.cam, dtype=np.float64), np.ascontiguousarray(prob.Xw, dtype=np.float64),
            np.ascontiguousarray(prob.idx2, dtype=np.int32), np.ascontiguousarray(prob.meas2, dtype=np.float64),
            np.ascontiguousarray(prob.omega2, dtype=np.float64), np.ascontiguousarray(prob.idx3, dtype=np.int32),
            np.ascontiguousarray(prob.meas3, dtype=np.float64), np.ascontiguousarray(prob.omega3, dtype=np.float64)]
    P = _Problem(prob.Pall, prob.numP, prob.Lall, prob.numL, _p(keep[0]), _p(keep[1]), _p(keep[2]), _p(keep[3]),
                 prob.E2, _p(keep[4]), _p(keep[5]), _p(keep[6]), prob.E3, _p(keep[7]), _p(keep[8]), _p(keep[9]))
    return P, keep


def transfer_bytes():
    """(h2d, d2h) bytes copied so far by this thread's engines"""
    a, b = C.c_longlong(0), C.c_longlong(0)
    _check(load_library().cuba_get_transfer_bytes(C.byref(a), C.byref(b)))
    return a.value, b.value


def build_structure_host(prob, rank=0, world=1):
    """Host-only structure build (no GPU needed): dict of index arrays + sizes."""
    L = load_library()
    P, keep = _problem_struct(prob)
    sz = _Sizes()
    _check(L.cuba_debug_build_structure_host(C.byref(P), rank, world, C.byref(sz), None, None, None, None, None, None, None, None))
    out = {n: getattr(sz, n) for n, _ in _Sizes._fields_}
    arrs = {"hplColPtr": np.zeros(sz.numL + 1, np.int32), "hplRowInd": np.zeros(sz.nhpl, np.int32),
            "edge2Hpl": np.zeros(sz.E2 + sz.E3, np.int32), "hscRowPtr": np.zeros(sz.numP + 1, np.int32),
            "hscColInd": np.zeros(sz.nblk, np.int32), "fullRowPtr": np.zeros(sz.numP + 1, np.int32),
            "fullColInd": np.zeros(sz.nblk_full, np.int32), "shard": np.zeros(4, np.int32)}
    _check(L.cuba_debug_build_structure_host(C.byref(P), rank, world, C.byref(sz), *[_p(arrs[k]) for k in
           ("hplColPtr", "hplRowInd", "edge2Hpl", "hscRowPtr", "hscColInd", "fullRowPtr", "fullColInd", "shard")]))
    out.update(arrs)
    return out


def pcg_partition_host(prob, n_ctas=148, max_aggregates=74):
    """Host side of the PCG setup on the CPU (row partition over n_ctas persistent CTAs, need lists, pose aggregates and coarse
    lists of the two-level PCG); the library verifies their invariants and raises CubaError if one fails."""
    L = load_library()
    P, keep = _problem_struct(prob)
    info = np.zeros(8, np.int32)
    _check(L.cuba_debug_pcg_partition(C.byref(P), int(n_ctas), int(max_aggregates), _p(info)))
    return dict(zip(("G", "gs", "A", "needMax", "maxRows", "blkMax", "maxNeedAgg", "coarse_list_size"), (int(v) for v in info)))


def pcg5_plan_host(prob, world=1, num_sms=148, max_aggregates=74):
    """Plan of the row-distributed two-level PCG on the CPU (rows over world x G virtual CTAs, rank-aligned aggregates, halo masks);
    the library verifies its invariants and raises CubaError if one fails."""
    L = load_library()
    P, keep = _problem_struct(prob)
    info = np.zeros(8, np.int32)
    _check(L.cuba_debug_pcg5_plan(C.byref(P), int(world), int(num_sms), int(max_aggregates), _p(info)))
    return dict(zip(("ok", "G", "gs", "A", "needMax", "maxRows", "maxNeedAgg", "halo_rows"), (int(v) for v in info)))


class Engine:
    """One optimizer instance on one GPU (reference: one CudaBundleAdjustment per thread/device)."""

    def __init__(self, device=-1, use_fp32=False, pcg_max_iters=0, pcg_tol=0.0, pcg_variant=0, structure_on_host=False, jh_variant=0,
                 coarse_refresh=0, two_level_switch=0, max_aggregates=0):
        self.L = load_library()
        res = (C.c_int * 7)()
        res[0] = int(pcg_variant)
        res[1] = int(bool(structure_on_host))
        res[2] = int(jh_variant)
        res[4] = int(coarse_refresh)
        res[5] = int(two_level_switch)
        res[6] = int(max_aggregates)
        cfg = _Config(device, 2 if use_fp32 == "mixed" else int(use_fp32), int(pcg_max_iters), float(pcg_tol), 1, res)
        h = C.c_void_p()
        _check(self.L.cuba_engine_create(C.byref(cfg), C.byref(h)))
        self.h = h
        self.sizes = None
        self._stats = []

    def close(self):
        if getattr(self, "h", None):
            self.L.cuba_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # --- reference API mirror ------------------------------------------------------------------------
    def set_robust_kernels(self, kernel_type, delta, edge_type):
        """setRobustKernels(kernelType, delta, edgeType), include/cuda_bundle_adjustment.h:93"""
        _check(self.L.cuba_engine_set_robust_kernel(self.h, int(edge_type), int(kernel_type), float(delta)))

    def set_comm(self, rank, world, unique_id=None):
        buf = None if unique_id is None else (C.c_char * 128).from_buffer_copy(bytes(unique_id))
        _check(self.L.cuba_engine_set_comm(self.h, rank, world, buf))

    @staticmethod
    def comm_unique_id():
        buf = (C.c_char * 128)()
        _check(load_library().cuba_comm_unique_id(buf))
        return bytes(buf)

    def initialize(self, prob):
        """initialize() + buildStructure(): upload the flat problem, build all index structures."""
        P, keep = _problem_struct(prob)
        _check(self.L.cuba_engine_set_problem(self.h, C.byref(P)))
        sz = _Sizes()
        _check(self.L.cuba_engine_get_sizes(self.h, C.byref(sz)))
        self.sizes = {n: getattr(sz, n) for n, _ in _Sizes._fields_}
        self._stats = []
        return self.sizes

    def set_structure_reuse(self, enable):
        _check(self.L.cuba_engine_set_structure_reuse(self.h, int(bool(enable))))

    def structure_reuses(self):
        n = C.c_longlong(0)
        _check(self.L.cuba_engine_get_structure_reuses(self.h, C.byref(n)))
        return n.value

    def set_state(self, q, t, Xw):
        q, t, Xw = (np.ascontiguousarray(a, dtype=np.float64) for a in (q, t, Xw))
        _check(self.L.cuba_engine_set_state(self.h, _p(q), _p(t), _p(Xw)))

    def reset_state(self):
        _check(self.L.cuba_engine_reset_state(self.h))

    def stream_ptr(self):
        s = C.c_void_p()
        _check(self.L.cuba_engine_get_stream(self.h, C.byref(s)))
        return s.value or 0

    def flush_l2(self):
        _check(self.L.cuba_engine_flush_l2(self.h))

    def optimize(self, niterations):
        stats = (_IterStat * max(niterations, 1))()
        n = C.c_int(0)
        _check(self.L.cuba_engine_optimize(self.h, niterations, stats, C.byref(n)))
        self._stats = [dict(iteration=s.iteration, trials=s.trials, chi2=s.chi2, lambda_=s.lambda_, pcg_iters=s.pcg_iters,
                            pcg_failed=s.pcg_failed) for s in stats[:n.value]]
        return self._stats

    def batch_statistics(self):
        return [(s["iteration"], s["chi2"]) for s in self._stats]

    def time_profile(self):
        sec = np.zeros(len(PROFILE_ITEMS))
        _check(self.L.cuba_engine_get_profile(self.h, _p(sec)))
        return dict(zip(PROFILE_ITEMS, sec.tolist()))

    def state(self):
        s = self.sizes
        q = np.zeros((s["Pall"], 4)); t = np.zeros((s["Pall"], 3)); Xw = np.zeros((s["Lall"], 3))
        _check(self.L.cuba_engine_get_state(self.h, _p(q), _p(t), _p(Xw)))
        return q, t, Xw

    def chi_squared(self):
        out = np.zeros(self.sizes["E2"] + self.sizes["E3"])
        _check(self.L.cuba_engine_get_chi2(self.h, _p(out)))
        return out

    def launch_count(self):
        n = C.c_longlong(0)
        _check(self.L.cuba_engine_get_launch_count(self.h, C.byref(n)))
        return n.value

    # --- stages ----------------------------------------------------------------------------------------
    def linearize(self):
        v = C.c_double(0)
        _check(self.L.cuba_stage_linearize(self.h, C.byref(v)))
        return v.value

    def max_diagonal(self):
        v = C.c_double(0)
        _check(self.L.cuba_stage_max_diagonal(self.h, C.byref(v)))
        return v.value

    def solve(self, lam):
        it, ok = C.c_int(0), C.c_int(0)
        _check(self.L.cuba_stage_solve(self.h, float(lam), C.byref(it), C.byref(ok)))
        return it.value, bool(ok.value)

    def update(self, lam):
        chi, sc = C.c_double(0), C.c_double(0)
        _check(self.L.cuba_stage_update(self.h, float(lam), C.byref(chi), C.byref(sc)))
        return chi.value, sc.value

    def commit(self, accept):
        _check(self.L.cuba_stage_commit(self.h, int(bool(accept))))

    def chi2(self):
        v = C.c_double(0)
        _check(self.L.cuba_stage_chi2(self.h, C.byref(v)))
        return v.value

    # --- debug -----------------------------------------------------------------------------------------
    def hpl_structure(self):
        s = self.sizes
        colPtr = np.zeros(s["numL"] + 1, np.int32); rowInd = np.zeros(s["nhpl"], np.int32); e2h = np.zeros(s["E2"] + s["E3"], np.int32)
        _check(self.L.cuba_debug_get_hpl_structure(self.h, _p(colPtr), _p(rowInd), _p(e2h)))
        return colPtr, rowInd, e2h

    def hsc_structure(self):
        s = self.sizes
        rowPtr = np.zeros(s["numP"] + 1, np.int32); colInd = np.zeros(s["nblk"], np.int32)
        _check(self.L.cuba_debug_get_hsc_structure(self.h, _p(rowPtr), _p(colInd)))
        return rowPtr, colInd

    def system(self):
        s = self.sizes
        Hpp = np.zeros((s["numP"], 36)); bp = np.zeros((s["numP"], 6)); Hll = np.zeros((s["numL"], 9)); bl = np.zeros((s["numL"], 3))
        Hpl = np.zeros((s["nhpl"], 18))
        _check(self.L.cuba_debug_get_system(self.h, _p(Hpp), _p(bp), _p(Hll), _p(bl), _p(Hpl)))
        return Hpp, bp, Hll, bl, Hpl

    def schur(self):
        s = self.sizes
        Hsc = np.zeros((s["nblk"], 36)); bsc = np.zeros((s["numP"], 6)); inv = np.zeros((s["numL"], 9))
        _check(self.L.cuba_debug_get_schur(self.h, _p(Hsc), _p(bsc), _p(inv)))
        return Hsc, bsc, inv

    def delta(self):
        s = self.sizes
        xp = np.zeros((s["numP"], 6)); xl = np.zeros((s["numL"], 3))
        _check(self.L.cuba_debug_get_delta(self.h, _p(xp), _p(xl)))
        return xp, xl

    def bench_stage(self, stage, reps=10, flush_l2=True, lam=1.0):
        ms = C.c_double(0)
        _check(self.L.cuba_bench_stage(self.h, int(stage), int(reps), int(bool(flush_l2)), float(lam), C.byref(ms)))
        return ms.value
