"""Writes tests/golden/score_order_ndt.npz: computeDerivatives, computeHessian, align and getFitnessScore of the CUDA engine
on the scene of tests/test_gpu_score_order.py.  The per-yaw source orderings feed the score kernel only, so these results
must stay bit-identical to the build that wrote the file (run it with B200REG_LIB pointing at that build).

    B200REG_LIB=/path/to/libb200reg.so python tools/make_score_order_golden.py [OUT.npz]
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

DELTAS = np.array([[0, 0, 0, 0, 0, 0], [0.12, -0.08, 0.03, 0.004, -0.006, 0.01], [0.4, 0.3, -0.1, 0.02, 0.03, -0.05]])
STARTS = np.array([[0.05, -0.04, 0.02, 0.0, 0.0, 0.005], [0.3, -0.25, 0.0, 0.0, 0.0, 0.035]])
FIT = np.array([[0, 0, 0, 0, 0, 0], [0.4, -0.3, 0.1, 0.01, 0.02, 0.05], [30.0, 5.0, 2.0, 0, 0, 1.0]])


def scene(synth):
    world = synth.make_world(synth.SEED, beams=True)
    mp = synth.sample_map(300_000, synth.SEED, world=world)
    p_true = np.array([3.0, -2.0, 1.2, 0.0, 0.0, 0.6])
    T = synth.pose_vec_to_matrix(p_true)
    dirs = synth.livox_dirs(5000, synth.SEED)
    scan = np.ascontiguousarray(synth.raycast(T[:3, 3], T[:3, :3], dirs, world, seed=synth.SEED)[:4000])
    return mp, scan, p_true


def compute(api, synth):
    mp, scan, p_true = scene(synth)
    out = {}
    for search in (1, 7, 27):
        g = api.NormalDistributionsTransform()
        g.setNeighborhoodSearchMethod(search)
        g.setTransformationEpsilon(0.01)
        g.setInputTarget(mp)
        g.setInputSource(scan)
        d = [g.computeDerivatives(p_true + dp) for dp in DELTAS]
        out[f"deriv_s_{search}"] = np.array([x[0] for x in d])
        out[f"deriv_g_{search}"] = np.stack([x[1] for x in d])
        out[f"deriv_H_{search}"] = np.stack([x[2] for x in d])
        out[f"hess_{search}"] = g.computeHessian(p_true + DELTAS[1])
        T, it = [], []
        for st in STARTS:
            g.align(synth.pose_vec_to_matrix(p_true + st).astype(np.float32))
            T.append(g.getFinalTransformation())
            it.append([g.result.iters, g.result.evals, g.result.hess_evals])
        out[f"align_T_{search}"] = np.stack(T)
        out[f"align_counts_{search}"] = np.array(it)
        out[f"fitness_{search}"] = np.array([g.getFitnessScore(T=synth.pose_vec_to_matrix(p_true + f).astype(np.float32)) for f in FIT])
        g.close()
    return out


if __name__ == "__main__":
    from pointcloud_slam_b200 import api, synth
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "score_order_ndt.npz")
    np.savez_compressed(path, **compute(api, synth))
    print("wrote", path, "from", api.lib_path())
