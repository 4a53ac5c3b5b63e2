"""Relocalization with NDT refinement (b200_reloc_refine) on one GPU: the candidates are the top K of calculateScore, every
candidate's refined record is bit-identical whatever else is in the call, it agrees with b200_ndt_align / the fitness call /
the oracle, and the refined winner is better than the grid's."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

OFFSET = np.array([0.2, -0.15, 0.0, 0.0, 0.0, 0.03])   # the grid's centre is off the truth: no hypothesis sits on it


@pytest.fixture(scope="module")
def scene(synth):
    world = synth.make_world(synth.SEED, beams=True)
    mp = synth.sample_map(300_000, synth.SEED, world=world)
    p_true = np.array([3.0, -2.0, 1.2, 0.0, 0.0, 0.6])
    T = synth.pose_vec_to_matrix(p_true)
    scan = np.ascontiguousarray(synth.raycast(T[:3, 3], T[:3, :3], synth.livox_dirs(5000, synth.SEED), world, seed=synth.SEED)[:4000])
    grid = synth.hypothesis_grid(p_true + OFFSET, nx=6, ny=6, nyaw=4, pitch=0.5)   # 144 hypotheses, 0.5 m apart
    return dict(map=mp, scan=scan, p_true=p_true, grid=grid)


@pytest.fixture(scope="module")
def ndt(api, scene):
    g = api.NormalDistributionsTransform()
    g.setTransformationEpsilon(0.01)
    g.setInputTarget(scene["map"])
    g.setInputSource(scene["scan"])
    return g


@pytest.fixture(scope="module")
def tied_grid(ndt, scene):
    """The grid with its best-scoring pose appended again: two hypotheses share the top score."""
    s = ndt.calculateScore(scene["grid"])
    return np.ascontiguousarray(np.concatenate([scene["grid"], scene["grid"][int(np.argmax(s))][None]], 0))


def refined_bytes(c):
    return bytes(c.refined)


def guess_of(pose16):
    return np.asarray(pose16, np.float32).reshape(4, 4).T


def test_candidates_are_the_top_k_scores(api, ndt, tied_grid):
    scores = ndt.calculateScore(tied_grid)
    keys = [api.score_key(float(s)) for s in scores]
    order = sorted(range(len(scores)), key=lambda i: (-keys[i], i))[:16]
    best, cands, ms = api.relocalize_refine(ndt, tied_grid, top_k=16)
    assert [c.hypothesis for c in cands] == order
    assert [c.initial_score for c in cands] == [scores[i] for i in order]       # the bits b200_ndt_score_batch returns
    dup = len(tied_grid) - 1
    assert order[1] == dup and order[0] < dup                                    # the tie: the lower index first
    assert refined_bytes(cands[0]) == refined_bytes(cands[1])                    # the same pose refines to the same bits
    assert cands.status in (0, 2) and best in order and ms > 0
    for c in cands.records[16:]:
        assert c.hypothesis == -1


def test_records_are_bit_identical_whatever_else_is_in_the_call(api, ndt, tied_grid):
    _, c16, _ = api.relocalize_refine(ndt, tied_grid, top_k=16)
    by_hyp = {c.hypothesis: refined_bytes(c) for c in c16}
    _, c4, _ = api.relocalize_refine(ndt, tied_grid, top_k=4)
    assert [refined_bytes(c) for c in c4] == [refined_bytes(c) for c in c16[:4]]
    for c in c16:                                                                # the pose alone, top_k = 1
        _, one, _ = api.relocalize_refine(ndt, tied_grid[c.hypothesis][None], h_begin=c.hypothesis, top_k=1)
        assert len(one) == 1 and one[0].hypothesis == c.hypothesis
        assert refined_bytes(one[0]) == by_hyp[c.hypothesis], c.hypothesis
        assert one[0].initial_score == c.initial_score
    for start in (0, 1):                                                         # interleaved slices on one GPU
        _, part, _ = api.relocalize_refine(ndt, tied_grid[start::2], h_begin=start, h_stride=2, top_k=16)
        assert all(c.hypothesis % 2 == start for c in part)
        for c in part:
            if c.hypothesis in by_hyp:
                assert refined_bytes(c) == by_hyp[c.hypothesis], c.hypothesis


def test_against_the_single_align_and_fitness(api, ndt, tied_grid):
    _, cands, _ = api.relocalize_refine(ndt, tied_grid, top_k=8, max_range=1.0)
    for c in cands[:4]:
        r = c.refined
        rc = ndt.align(guess_of(tied_grid[c.hypothesis]))
        s = ndt.result
        assert (r.ndt.iters, r.ndt.evals, r.ndt.converged) == (s.iters, s.evals, s.converged)
        assert r.status == rc
        final = np.array(r.final16, np.float32).reshape(4, 4).T
        np.testing.assert_allclose(final, ndt.getFinalTransformation(), atol=1e-6)
        assert abs(r.ndt.trans_probability - s.trans_probability) <= 1e-6 * abs(s.trans_probability)
        assert ndt.getFitnessScore(1.0, T=final) == r.fitness and ndt.fitness_in_range == r.n_in_range


def test_top_candidates_match_the_oracle(oracle, api, ndt, scene, tied_grid):
    o = oracle.OracleNdt(resolution=1.0, trans_eps=0.01)
    o.set_target(scene["map"])
    o.set_source(scene["scan"])
    _, cands, _ = api.relocalize_refine(ndt, tied_grid, top_k=8)
    for c in cands[:3]:
        rc, T0, r0 = o.align(guess_of(tied_grid[c.hypothesis]))
        assert c.refined.ndt.iters == r0.iters and c.refined.status == rc
        dp = np.array(c.refined.ndt.p_final) - np.array(r0.p_final)
        assert np.abs(dp[:3]).max() < 1e-4 and np.abs(dp[3:]).max() < 1e-4


def test_refined_winner_beats_the_grid(oracle, api, ndt, scene):
    grid, p_true = scene["grid"], scene["p_true"]
    arg, _, _ = api.relocalize(ndt, grid)
    assert np.linalg.norm(guess_of(grid[arg])[:3, 3] - p_true[:3]) >= 0.1   # the score-only winner is a grid point
    best, cands, _ = api.relocalize_refine(ndt, grid, top_k=16)
    assert cands.status == 0
    w = next(c for c in cands if c.hypothesis == best)
    assert w.refined.status == 0 and w.refined.ndt.converged
    o = oracle.OracleNdt(resolution=1.0, trans_eps=0.01)
    o.set_target(scene["map"])
    o.set_source(scene["scan"])
    rc, T0, r0 = o.align(guess_of(grid[best]))
    dp = np.array(w.refined.ndt.p_final) - np.array(r0.p_final)
    assert rc == 0 and np.abs(dp[:3]).max() < 1e-2 and np.abs(dp[3:]).max() < 1e-3
    assert np.abs(np.array(w.refined.ndt.p_final)[:3] - p_true[:3]).max() < 0.1


def test_edges(api, ndt, scene):
    grid = scene["grid"]
    ERR_ARG, NO_POINTS = -1, 1
    arg0 = api.relocalize(ndt, grid)[:2]
    # top_k beyond the hypotheses with a finite score; a NaN pose is never a candidate
    few = grid[:5].copy()
    few[2, 12] = np.nan
    best, cands, _ = api.relocalize_refine(ndt, few, top_k=64)
    assert len(cands) == 4 and 2 not in [c.hypothesis for c in cands]
    assert all(c.hypothesis == -1 for c in cands.records[4:])
    # no hypothesis on the only GPU
    best, cands, _ = api.relocalize_refine(ndt, np.zeros((0, 16), np.float32), top_k=4)
    assert (best, cands.status, len(cands)) == (-1, NO_POINTS, 0)
    # malformed calls
    import ctypes
    lib = api.lib()
    res = (api.RelocCandidate * 4)()
    b, nc = ctypes.c_int64(0), ctypes.c_int64(0)
    p = api._p(np.ascontiguousarray(grid[:4]))
    h = ndt._handle()
    call = lambda *a: lib.b200_reloc_refine(None, *a)
    assert call(h, p, 4, 0, 1, 0, 1.0, ctypes.byref(b), res, ctypes.byref(nc), None) == ERR_ARG          # top_k = 0
    assert call(h, p, 4, 0, 1, 65536, 1.0, ctypes.byref(b), res, ctypes.byref(nc), None) == ERR_ARG      # top_k too large
    assert call(h, p, -1, 0, 1, 4, 1.0, ctypes.byref(b), res, ctypes.byref(nc), None) == ERR_ARG         # h < 0
    assert call(h, None, 4, 0, 1, 4, 1.0, ctypes.byref(b), res, ctypes.byref(nc), None) == ERR_ARG       # h > 0, no poses
    assert call(h, p, 4, 0, 0, 4, 1.0, ctypes.byref(b), res, ctypes.byref(nc), None) == ERR_ARG          # stride 0
    assert call(h, p, 4, 0, 1, 4, 1.0, None, res, ctypes.byref(nc), None) == ERR_ARG                     # no best
    assert call(h, p, 4, 0, 1, 4, 1.0, ctypes.byref(b), None, ctypes.byref(nc), None) == ERR_ARG         # no cands
    bare = api.NormalDistributionsTransform()
    bare.setInputTarget(scene["map"])
    assert call(bare._handle(), p, 4, 0, 1, 4, 1.0, ctypes.byref(b), res, ctypes.byref(nc), None) == ERR_ARG   # no source
    assert b"no source" in lib.b200_last_error()
    bare.close()
    # the score-only relocalization is unchanged around it
    assert api.relocalize(ndt, grid)[:2] == arg0


def test_refine_adaptor_on_gpu(tmp_path, api):
    from test_reloc_refine_cpu import build_adaptor
    exe = build_adaptor(tmp_path, api)
    p = subprocess.run([exe], capture_output=True, text=True, timeout=300, cwd=ROOT, env=dict(os.environ))
    assert p.returncode == 0 and "relocalization adaptor ok" in p.stdout, p.stdout + p.stderr
