"""The LOAM oracle (fp32, the device's operation order) against an independent fp64 restatement (tests/loam_ref.py): feature
flags and coefficients, the first A^T A against a central-difference Jacobian, the degeneracy projection of the LM step and the
5-NN range gate.  With the device-to-oracle bit parity of the GPU tests this ties the device to fp64 math: an error the
device and the oracle share (a wrong Jacobian row, the wrong eigenvector, a wrong projection) fails here."""
import numpy as np
import pytest

import loam_ref as lr

POSES = ((0.01, -0.02, 0.6, 3.0, -2.0, 1.2),) + lr.LARGE_ANGLE_POSES
GUESS = np.array([0.01, -0.01, 0.02, 0.15, -0.1, 0.05], np.float32)


@pytest.fixture(scope="module", params=POSES, ids=lambda t: "rpy=%g,%g,%g" % t[:3])
def posed(request, oracle, synth):
    sc = synth.loam_scene(t_true=request.param)
    o = oracle.OracleLoam()
    o.set_map(sc["corner_map"], sc["surf_map"])
    return sc, o


@pytest.fixture(scope="module")
def corridor(oracle):
    sc = lr.corridor()
    o = oracle.OracleLoam()
    o.set_map(sc["corner_map"], sc["surf_map"])
    return sc, o


def check_pass(sc, o, t6):
    n, flags, coeff = o.features(sc["corner"], sc["surf"], t6)
    ref = lr.Pass(sc["corner_map"], sc["surf_map"], sc["corner"], sc["surf"], t6)
    both = lr.check_features(ref, flags, coeff)
    assert both.sum() > 0.8 * flags.sum()
    return flags, coeff


def test_features_match_fp64(posed):
    sc, o = posed
    for t6 in (sc["t_true"], sc["t_true"] + GUESS):
        check_pass(sc, o, t6)


def test_first_normal_matrix_matches_fp64_jacobian(posed):
    sc, o = posed
    guess = sc["t_true"] + GUESS
    flags, coeff = check_pass(sc, o, guess)
    _, st = o.optimize(sc["corner"], sc["surf"], guess, iter_num=1)
    assert lr.rel_err(st["AtA"], lr.jtj(sc["corner"], sc["surf"], flags, coeff, guess)) <= 1e-5


def test_corridor_is_degenerate_and_the_step_avoids_the_weak_direction(corridor):
    sc, o = corridor
    guess = sc["t_true"] + GUESS
    flags, coeff = check_pass(sc, o, guess)
    t1, st = o.optimize(sc["corner"], sc["surf"], guess, iter_num=1)
    assert lr.rel_err(st["AtA"], lr.jtj(sc["corner"], sc["surf"], flags, coeff, guess)) <= 1e-5
    lam = np.linalg.eigvalsh(st["AtA"])
    assert st["degenerate"] and lam[0] < 100 < lam[1]
    assert lr.weak_step_fraction(st["AtA"], guess, t1) <= 1e-5
    # the weak direction is x (along the corridor): the offset along it is never corrected
    t, st = o.optimize(sc["corner"], sc["surf"], guess)
    assert st["converged"] and st["degenerate"]
    assert abs(t[3] - guess[3]) < 1e-3 and np.abs(t[[4, 5]] - sc["t_true"][[4, 5]]).max() < 1e-3


def test_range_gate_is_strict_and_exact(oracle):
    surf_map, scan = lr.lattice()
    d5 = np.array([np.sort(lr.fp32_d2(surf_map, q))[4] for q in scan])
    assert d5[0] == np.float32(1.0) and d5[1] == np.nextafter(np.float32(1), np.float32(0))
    o = oracle.OracleLoam()
    o.set_map(np.zeros((0, 3), np.float32), surf_map)
    n, flags, coeff = o.features(np.zeros((0, 3), np.float32), scan, np.zeros(6, np.float32))
    np.testing.assert_array_equal(flags[:3], (d5[:3] < 1.0).astype(np.uint8))    # [0, 1, 1]
    np.testing.assert_array_equal(flags[:3], [0, 1, 1])
    # on the plane z = 5 the coefficient is (0, 0, +-1, pd2 = 0) with weight 1
    np.testing.assert_allclose(np.abs(coeff[1:3]), [[0, 0, 1, 0]] * 2, atol=1e-6)
