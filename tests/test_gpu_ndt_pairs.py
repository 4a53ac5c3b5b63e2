"""Batched NDT registration of independent (source, target) pairs (b200_ndt_pairs_align) against the CPU oracle, the
single-pair device path, itself (determinism across batch composition and chunking) and the synthetic ground truth.

Bars: leaves bit-exact; align as test_gpu_ndt.test_align_parity (rc / converged / iteration counts equal, p_final within
1e-4, trans_probability within 1e-6 relative); fitness within 1e-12 relative of the oracle and bit-equal to
b200_ndt_fitness_score at the same transformation; finals within 1e-6 of b200_ndt_align (test_align_batch_equals_single).
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

N_SRC = [500, 15000, 2000, 8000, 1200, 12000, 4000, 700, 10000, 3000, 6000, 900,
         14000, 2500, 5000, 800, 9000, 1500, 11000, 3500, 600, 7000, 13000, 1800]
N_TGT = [20000, 150000, 60000, 100000, 30000, 120000, 45000, 25000, 90000, 70000, 80000, 35000,
         140000, 50000, 65000, 22000, 110000, 40000, 130000, 55000, 28000, 75000, 95000, 33000]
SETTINGS = dict(resolution=1.0, trans_eps=0.01, step_size=0.1, max_iter=35)


@pytest.fixture(scope="module")
def pairs(synth):
    return synth.loop_pairs(len(N_SRC), N_SRC, N_TGT)


def run_batch(api, d, search=7, order=None, max_range=1.7976931348623157e308):
    order = list(range(len(d["sources"]))) if order is None else list(order)
    b = api.NdtPairBatch(search=search, **SETTINGS)
    r = b.align([d["sources"][i] for i in order], [d["targets"][i] for i in order], max_range=max_range)
    return b, r


def record_bytes(r, k):
    rec = type(r["records"][0]).from_buffer_copy(r["records"][k])
    rec.ndt.gpu_ms = 0.0   # device time of the call is the only field that may differ
    return bytes(memoryview(rec).cast("B"))


def oracle_for(oracle, d, p, search=7):
    o = oracle.OracleNdt(search=search, **SETTINGS)
    o.set_target(d["targets"][p])
    o.set_source(d["sources"][p])
    return o


def test_leaves_bit_exact(oracle, api, pairs):
    b, r = run_batch(api, pairs)
    assert (r["status"] == 0).all()
    for p in range(len(N_SRC)):
        o = oracle_for(oracle, pairs, p)
        Lo, Lg = o.leaves(), b.leaves(p)
        for k in ("ids", "npts", "mean", "cov", "icov"):
            np.testing.assert_array_equal(Lg[k], Lo[k], err_msg=f"pair {p} {k}")


@pytest.mark.parametrize("search", [7, 1, 0])
def test_align_and_fitness_vs_oracle(oracle, api, pairs, search):
    sel = range(len(N_SRC)) if search == 7 else range(0, len(N_SRC), 3)
    _, r = run_batch(api, pairs, search=search)
    _, rs = run_batch(api, pairs, search=search, max_range=0.05)
    for p in sel:
        o = oracle_for(oracle, pairs, p, search)
        rc0, T0, r0 = o.align(np.eye(4, dtype=np.float32))
        assert r["status"][p] == rc0 and r["converged"][p] == r0.converged, p
        assert (r["iters"][p], r["evals"][p], r["hess_evals"][p]) == (r0.iters, r0.evals, r0.hess_evals), p
        assert np.abs(r["p_final"][p] - np.array(r0.p_final)).max() < 1e-4, p
        assert abs(r["trans_probability"][p] - r0.trans_probability) <= 1e-6 * abs(r0.trans_probability), p
        for res, mr in ((r, 1.7976931348623157e308), (rs, 0.05)):
            s0, n0 = o.fitness(res["final"][p], max_range=mr)
            assert res["n_in_range"][p] == n0, p
            assert abs(res["fitness"][p] - s0) <= 1e-12 * abs(s0) or (n0 == 0 and res["fitness"][p] == s0), p


def test_equals_single_pair_path(api, pairs):
    _, r = run_batch(api, pairs)
    _, rs = run_batch(api, pairs, max_range=0.05)
    for p in range(len(N_SRC)):
        g = api.NormalDistributionsTransform()
        g.setTransformationEpsilon(SETTINGS["trans_eps"])
        g.setInputTarget(pairs["targets"][p])
        g.setInputSource(pairs["sources"][p])
        rc = g.align(None)
        assert rc == r["status"][p]
        assert (g.result.iters, g.result.evals, g.result.converged) == (r["iters"][p], r["evals"][p], r["converged"][p]), p
        np.testing.assert_allclose(r["final"][p], g.getFinalTransformation(), atol=1e-6)
        # getFitnessScore at the batch's own final transformation: the same bits as the single-target kernel
        assert g.getFitnessScore(T=r["final"][p]) == r["fitness"][p] and g.fitness_in_range == r["n_in_range"][p], p
        assert g.getFitnessScore(max_range=0.05, T=rs["final"][p]) == rs["fitness"][p], p


def test_ground_truth(oracle, api, pairs):
    """The final transformation undoes the synthetic drift as well as the oracle's own does."""
    _, r = run_batch(api, pairs)
    for p in range(0, len(N_SRC), 2):
        _, T0, _ = oracle_for(oracle, pairs, p).align(np.eye(4, dtype=np.float32))
        Tt = pairs["T_true"][p]
        e_dev = np.abs(r["final"][p][:3, 3] - Tt[:3, 3]).max()
        e_orc = np.abs(T0[:3, 3] - Tt[:3, 3]).max()
        assert e_dev <= e_orc + 1e-4, (p, e_dev, e_orc)
        yaw = lambda M: np.arctan2(M[1, 0], M[0, 0])
        assert abs(yaw(r["final"][p]) - yaw(Tt)) <= abs(yaw(T0) - yaw(Tt)) + 1e-4, p


def test_determinism_across_batches_and_chunks(api, pairs, tmp_path):
    """Every pair's record is bit-identical alone, in the full batch, in a shuffled batch and with 5 pairs per chunk."""
    P = len(N_SRC)
    _, full = run_batch(api, pairs)
    perm = np.random.default_rng(3).permutation(P)
    _, shuf = run_batch(api, pairs, order=perm)
    for k, p in enumerate(perm):
        assert record_bytes(shuf, k) == record_bytes(full, p), p
    for p in (0, 1, 7, 12):
        _, alone = run_batch(api, pairs, order=[p])
        assert record_bytes(alone, 0) == record_bytes(full, p), p
    # chunked run in a fresh process (the switch is read once per process)
    np.savez(tmp_path / "pairs.npz", **{f"s{p}": pairs["sources"][p] for p in range(P)}, **{f"t{p}": pairs["targets"][p] for p in range(P)})
    out = tmp_path / "chunked.bin"
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from pointcloud_slam_b200 import api; d = np.load(%r); P = %d; "
            "b = api.NdtPairBatch(search=7, **%r); r = b.align([d[f's{p}'] for p in range(P)], [d[f't{p}'] for p in range(P)]); "
            "open(%r, 'wb').write(b''.join(bytes(memoryview(r['records'][p]).cast('B')) for p in range(P)))"
            % (ROOT, str(tmp_path / "pairs.npz"), P, SETTINGS, str(out)))
    proc = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, B200_NDT_PAIRS_CHUNK="5"), capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr[-3000:]
    blob = out.read_bytes()
    n = ctypes.sizeof(full["records"][0])
    for p in range(P):
        rec = type(full["records"][0]).from_buffer_copy(blob[p * n:(p + 1) * n])
        rec.ndt.gpu_ms = 0.0
        assert bytes(memoryview(rec).cast("B")) == record_bytes(full, p), p


def test_isolation_of_bad_pairs(oracle, api, pairs):
    """An all-NaN target and a source that misses its target get the single path's statuses / iteration counts; the other
    pairs are bit-identical to a batch without them; an empty source is B200_ERR_ARG for that pair alone."""
    keep = [0, 2, 4, 6]
    _, clean = run_batch(api, pairs, order=keep)
    nan_tgt = np.full((5000, 3), np.nan, np.float32)
    far_src = pairs["sources"][2] + np.float32(500.0)
    srcs = [pairs["sources"][0], pairs["sources"][1], pairs["sources"][2], far_src, pairs["sources"][4], np.zeros((0, 3), np.float32),
            pairs["sources"][6]]
    tgts = [pairs["targets"][0], nan_tgt, pairs["targets"][2], pairs["targets"][2], pairs["targets"][4], pairs["targets"][5], pairs["targets"][6]]
    b = api.NdtPairBatch(search=7, **SETTINGS)
    r = b.align(srcs, tgts)
    # all-NaN target: what b200_ndt_set_target returns
    g = api.NormalDistributionsTransform()
    g.setInputTarget(nan_tgt)
    with pytest.raises(api.B200Error) as e:
        g.numVoxels()
    assert r["status"][1] == -1 and "no finite point" in str(e.value)
    assert b.leaves(1) is None
    # source outside the target: the oracle's early stop (zero step, converged)
    o = oracle_for(oracle, dict(sources=[far_src], targets=[pairs["targets"][2]]), 0)
    rc0, T0, r0 = o.align(np.eye(4, dtype=np.float32))
    assert (r["status"][3], r["iters"][3], r["evals"][3], r["converged"][3]) == (rc0, r0.iters, r0.evals, r0.converged)
    assert r["status"][5] == -1 and r["iters"][5] == 0
    for i, k in enumerate((0, 2, 4, 6)):   # batch positions of the healthy pairs
        assert record_bytes(r, k) == record_bytes(clean, i), k


def test_malformed_calls_fail_as_a_whole(api, pairs):
    b = api.NdtPairBatch()
    src, soff = b.pack(pairs["sources"][:2])
    tgt, toff = b.pack(pairs["targets"][:2])
    with pytest.raises(api.B200Error, match="offsets"):
        b.align_packed(src, soff[::-1].copy(), tgt, toff, 2)
    with pytest.raises(api.B200Error):
        b.align_packed(src, soff, tgt, toff, 0)


def test_cpp_adaptor_runs(tmp_path, api):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_ndt_pairs_cpu import build_adaptor
    p = subprocess.run([build_adaptor(tmp_path, api)], capture_output=True, text=True)
    assert p.returncode == 0 and "ndt pairs adaptor ok" in p.stdout, p.stdout + p.stderr
