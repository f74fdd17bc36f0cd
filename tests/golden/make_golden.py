"""Generates the committed golden fixtures from a checkout of the reference (needs its two vendored scans; no GPU):

    python tests/golden/make_golden.py <path of the lidarslam_ros2 checkout>

 * pcd_target_ds.npy / pcd_source_ds.npy: the two vendored scans of the reference
   (Thirdparty/ndt_omp_ros2/data/251370668.pcd = target, 251371071.pcd = source) after the 0.1 m VoxelGrid that
   apps/align.cpp:66-75 applies, produced by the ORACLE's pcl::VoxelGrid restatement. float32 xyz.
 * golden.json: the README's printed fitness values (Thirdparty/ndt_omp_ros2/README.md:19-52) — the only
   known-answer numbers in the reference — plus the oracle's poses / iteration counts for the same runs.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle  # noqa: E402
from lidarslam_ros2_b200.pcd import load_pcd  # noqa: E402

REF = os.path.join(sys.argv[1], "Thirdparty", "ndt_omp_ros2", "data", "")
tgt = load_pcd(REF + "251370668.pcd")
src = load_pcd(REF + "251371071.pcd")
tg = oracle.voxelgrid(tgt[:, :3], 0.1)[:, :3].copy()
sr = oracle.voxelgrid(src[:, :3], 0.1)[:, :3].copy()
np.save(os.path.join(HERE, "pcd_target_ds.npy"), tg)
np.save(os.path.join(HERE, "pcd_source_ds.npy"), sr)
# a raw 4-field slice (x, y, z, intensity) for the VoxelGrid all-fields test
np.save(os.path.join(HERE, "pcd_source_raw_head.npy"), src[:20000].copy())

readme = {"KDTREE": 0.213937, "DIRECT7": 0.214205, "DIRECT1": 0.208511, "GICP": 0.220388}
out = {"readme_fitness": readme, "n_target_ds": int(len(tg)), "n_source_ds": int(len(sr)), "ndt": {}}
for name, m in (("KDTREE", 0), ("DIRECT7", 2), ("DIRECT1", 3)):
    n = oracle.NDT(resolution=1.0, search_method=m)  # apps/align.cpp:90-104 defaults: eps 0.1, 35 its, step 0.1
    n.set_target(tg)
    n.set_source(sr)
    T = n.align()
    out["ndt"][name] = {
        "final_transformation": [[float(v) for v in row] for row in T],
        "iterations": n.iterations,
        "evaluations": n.evaluations,
        "converged": bool(n.converged),
        "fitness": n.fitness(),
        "trans_probability": n.trans_probability,
    }
    print(name, out["ndt"][name]["fitness"], "README", readme[name])
    assert abs(out["ndt"][name]["fitness"] - readme[name]) < 5e-6
with open(os.path.join(HERE, "golden.json"), "w") as f:
    json.dump(out, f, indent=1)
print("wrote golden fixtures")
