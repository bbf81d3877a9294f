#!/usr/bin/env python3
"""Generates tests/golden/kitti07_sub.npz and kitti00_sub.npz: small pieces of the reference's two real graphs
(ba_kitti_07, ba_kitti_00), so that the tests can run on real measurements without the full fixtures, which are
too large to store.  Needs oracle/_ref/fixtures (extracted by build() where the reference sources are present).

kitti07_sub: the first 20 poses, landmarks seen by at least two of them, a seeded sample of those.
kitti00_sub: the poses that see the most-observed landmark, the landmarks with more than 32 observations among
  them (the J+H kernels cut those into pieces) and a seeded sample of the others.
In both, the lowest pose id is fixed, like the first pose of the full graphs.  Floating-point arrays whose
values are all float32 numbers (the measurements and information weights of the fixtures) are stored as float32."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402


def _observations(g):
    return np.concatenate([g["mono_vP"], g["stereo_vP"]]), np.concatenate([g["mono_vL"], g["stereo_vL"]])


def subgraph(g, pose_ids, lm_ids):
    pose_ids, lm_ids = np.sort(pose_ids), np.sort(lm_ids)
    pm, lm = np.isin(g["pose_id"], pose_ids), np.isin(g["lm_id"], lm_ids)
    s = {k: g[k][pm] for k in ("pose_id", "pose_fixed", "q", "t", "cam")}
    s.update({k: g[k][lm] for k in ("lm_id", "lm_fixed", "Xw")})
    s["pose_fixed"] = (s["pose_id"] == s["pose_id"].min()).astype(np.int32)
    for kind in ("mono", "stereo"):
        em = np.isin(g[kind + "_vP"], pose_ids) & np.isin(g[kind + "_vL"], lm_ids)
        for k in ("vP", "vL", "meas", "info"):
            s["%s_%s" % (kind, k)] = g["%s_%s" % (kind, k)][em]
    return s


def kitti07_sub(g, rng):
    poses = np.sort(g["pose_id"])[:20]
    vP, vL = _observations(g)
    u, c = np.unique(vL[np.isin(vP, poses)], return_counts=True)
    lms = rng.choice(u[c >= 2], 450, replace=False)
    return subgraph(g, poses, lms)


def kitti00_sub(g, rng):
    vP, vL = _observations(g)
    u, c = np.unique(vL, return_counts=True)
    poses = np.unique(vP[vL == u[np.argmax(c)]])
    u, c = np.unique(vL[np.isin(vP, poses)], return_counts=True)
    big = u[c > 32]
    lms = np.concatenate([big[:8], rng.choice(u[(c >= 2) & (c <= 32)], 450, replace=False)])
    return subgraph(g, poses, lms)


def save(path, s):
    out = {}
    for k, a in s.items():
        if a.dtype == np.float64 and np.array_equal(a.astype(np.float32).astype(np.float64), a):
            a = a.astype(np.float32)
        out[k] = a
    np.savez_compressed(path, **out)
    print("wrote %s: %d poses %d landmarks %d mono %d stereo, %d bytes" % (path, len(s["pose_id"]), len(s["lm_id"]), len(s["mono_vP"]),
                                                                       len(s["stereo_vP"]), os.path.getsize(path)))


def main():
    pkg = ge.load_package()
    fx = os.path.join(ROOT, "oracle", "_ref", "fixtures")
    for name, fn, seed in (("kitti07_sub", kitti07_sub, 7), ("kitti00_sub", kitti00_sub, 0)):
        g = pkg.graphio.read_graph(os.path.join(fx, name.replace("_sub", "").replace("kitti", "ba_kitti_") + ".cubagraph"))
        save(os.path.join(HERE, name + ".npz"), fn(g, np.random.default_rng(seed)))


if __name__ == "__main__":
    main()
