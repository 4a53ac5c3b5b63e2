"""Worker of tests/test_gpu_loam_more.py: one process per candidate-walk variant of the LOAM search (B200_KNN_MODE is read
once per process).  Runs one features pass and one scan2MapOptimization on a sparse scene (60k-point surf map, ~2.5 points
per 1 m voxel) and a dense one (250k points, ~9 per voxel: more than 64 stencil candidates per query, beyond the flat list
of walk 5) and saves the results to the .npz named by argv[1]."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from pointcloud_slam_b200 import api  # noqa: E402
import loam_ref  # noqa: E402

out = {}
for name, sc in loam_ref.mode_scenes().items():
    g = api.ScanToMap(max_map_points=300_000)
    g.setInputCloud(sc["corner_map"], sc["surf_map"])
    n, flags, coeff = g.features(sc["corner"], sc["surf"], sc["guess"])
    t6, rc = g.scan2MapOptimization(sc["corner"], sc["surf"], sc["guess"])
    st = g.stats
    out[name + "_flags"], out[name + "_coeff"], out[name + "_t6"] = flags, coeff, t6
    out[name + "_stats"] = np.array([rc, st.iters, st.n_sel, st.converged, st.degenerate])
    out[name + "_AtA"] = np.array(st.AtA_first)
    g.close()
np.savez(sys.argv[1], **out)
