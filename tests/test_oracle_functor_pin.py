"""Pin of the oracle's restated cost functors against the REFERENCE's own functor text (round-1 verdict, item 8).

oracle/_ref/libref_functors.so is include/icp-ceres.h (all twelve functors) + include/eigen_quaternion.h compiled UNMODIFIED from
the reference tree against oracle/stubs/ (mini Eigen interface, Ceres class shells, three members of Sophus::SE3Group) and
differentiated with the oracle's Jet (oracle/ref_functors.cpp; recipe oracle/Makefile).  Its answers for the first iterations of
every loop below are stored in tests/golden/ref_pins.npz (tests/golden/make_golden.py:ref_pins) and always checked; the loops run
in full against the library wherever oracle/_ref was built.

Tolerance: the restatement and the reference text may associate 3-term sums differently (Eigen 3.3 reduces x0 + (x1 + x2),
the restatement folds left), so values are compared to a few ulps of the magnitudes that enter them, not bit for bit."""
import numpy as np
import pytest

EPS = np.finfo(np.float64).eps


def _rand_pose(rng, param, unit=True):
    if param == 0:
        return np.concatenate([rng.normal(0, 0.8, 3), rng.normal(0, 0.5, 3)])
    q = rng.normal(size=4)
    q /= np.linalg.norm(q)
    if not unit:
        q *= rng.uniform(0.98, 1.02)       # the reference runs its functors on non-unit quaternions too (non-rigid sample poses)
    return np.concatenate([q, rng.normal(0, 0.5, 3)])


@pytest.fixture(scope="module")
def pins(golden_dir):
    return np.load(f"{golden_dir}/ref_pins.npz")


def _split(x, *sizes):
    return np.split(x, np.cumsum(sizes)[:-1])


@pytest.mark.parametrize("param", [0, 1, 2])
@pytest.mark.parametrize("plane", [0, 1])
def test_global_functors_match_reference_text(oracle, pins, param, plane):
    G = 6 if param == 0 else 7
    k = f"gfun_p{param}_l{plane}"
    for x, r1, j1 in zip(pins[k + "_in"], pins[k + "_r"], pins[k + "_j"]):
        c1, c2, src, dst, nor = _split(x, G, G, 3, 3, 3)
        r0, j0 = oracle.functor_eval(param, plane, c1, c2, src, dst, nor, "oracle")
        scale = 1.0 + np.abs(c1).max() + np.abs(c2).max() + np.abs(src).max() + np.abs(dst).max()
        assert np.abs(r0 - r1).max() / scale <= 16 * EPS and np.abs(j0 - j1).max() / scale <= 32 * EPS
    if oracle.ref_functors() is None:
        return
    rng = np.random.default_rng(100 + 10 * param + plane)
    worst_r = worst_j = 0.0
    for it in range(10_000 // 6 + 1):
        c1 = _rand_pose(rng, param, unit=it % 3 != 0); c2 = _rand_pose(rng, param, unit=it % 3 != 0)
        if param == 0 and it % 50 == 0:
            c1[:3] = rng.normal(0, 1e-9, 3)     # first-order branch of AngleAxisRotatePoint (theta^2 <= DBL_EPSILON)
        src = rng.normal(0, 0.3, 3); dst = rng.normal(0, 0.3, 3); nor = rng.normal(size=3); nor /= np.linalg.norm(nor)
        r0, j0 = oracle.functor_eval(param, plane, c1, c2, src, dst, nor, "oracle")
        r1, j1 = oracle.functor_eval(param, plane, c1, c2, src, dst, nor, "ref")
        scale = 1.0 + np.abs(c1).max() + np.abs(c2).max() + np.abs(src).max() + np.abs(dst).max()
        worst_r = max(worst_r, np.abs(r0 - r1).max() / scale); worst_j = max(worst_j, np.abs(j0 - j1).max() / scale)
    assert worst_r <= 16 * EPS and worst_j <= 32 * EPS, (worst_r / EPS, worst_j / EPS)


@pytest.mark.parametrize("param", [0, 1, 2])
@pytest.mark.parametrize("plane", [0, 1])
def test_pairwise_functors_are_the_global_ones_with_identity_dst(oracle, pins, param, plane):
    """icp-ceres.h:320-552 (one pose) against the restated global functor with an identity dst pose -- the way the engine and the
    oracle run the pairwise solvers (a two-frame problem whose frame 0 is constant at identity)."""
    ident = np.zeros(6) if param == 0 else np.array([0, 0, 0, 1.0, 0, 0, 0])
    G = 6 if param == 0 else 7
    k = f"pfun_p{param}_l{plane}"
    for x, r1, j1 in zip(pins[k + "_in"], pins[k + "_r"], pins[k + "_j"]):
        c1, src, dst, nor = _split(x, G, 3, 3, 3)
        r0, j0 = oracle.functor_eval(param, plane, c1, ident, src, dst, nor, "oracle")
        assert np.abs(r0 - r1).max() <= 32 * EPS and np.abs(j0[:, :G] - j1).max() <= 64 * EPS
    if oracle.ref_functors() is None:
        return
    rng = np.random.default_rng(200 + 10 * param + plane)
    for it in range(1000):
        c1 = _rand_pose(rng, param)
        src = rng.normal(0, 0.3, 3); dst = rng.normal(0, 0.3, 3); nor = rng.normal(size=3); nor /= np.linalg.norm(nor)
        r0, j0 = oracle.functor_eval(param, plane, c1, ident, src, dst, nor, "oracle")
        r1, j1 = oracle.functor_eval_pairwise_ref(param, plane, c1, src, dst, nor)
        assert np.abs(r0 - r1).max() <= 32 * EPS and np.abs(j0[:, :G] - j1).max() <= 64 * EPS


def test_quaternion_parameterisation_matches_reference_text(oracle, pins):
    """eigen_quaternion.h:89-117: Plus (left-multiplied [sin|d| d/|d|, cos|d|], identity at d = 0) and the hand-written 4x3 Jacobian."""
    import ctypes as C
    P = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    for x, d, out, j in zip(pins["quat_x"], pins["quat_d"], pins["quat_plus"], pins["quat_jac"]):
        assert np.abs(out - oracle.quat_plus(x, d)).max() <= 8 * EPS
        j0 = np.zeros(12); oracle.lib().orc_quat_jacobian(P(np.ascontiguousarray(x)), P(j0))
        assert np.array_equal(j, j0)
    lib = oracle.ref_functors()
    if lib is None:
        return
    rng = np.random.default_rng(7)
    for it in range(2000):
        x = rng.normal(size=4); x /= np.linalg.norm(x)
        d = rng.normal(0, 0.3, 3) if it % 10 else np.zeros(3)
        out = np.zeros(4); lib.ref_quat_plus(P(x), P(d), P(out))
        assert np.abs(out - oracle.quat_plus(x, d)).max() <= 8 * EPS
        j = np.zeros(12); lib.ref_quat_jacobian(P(x), P(j))
        j0 = np.zeros(12); oracle.lib().orc_quat_jacobian(P(x), P(j0))
        assert np.array_equal(j, j0)
