"""The long-double Riccati / LQ reference (tests/lqref.py) against the pinned results of the parity tests
(tests/golden/expected/lq{r}_*.npz), on those tests' own seeded inputs.  The pins were checked against the original
discopt.dlqr run live, so this ties the reference to it; the GPU tests (test_gpu_riccati.py) then hold the kernels to
the reference at shapes the pins never covered.  CPU only."""
import numpy as np
import pytest

import golden_util as G
import lqref


def lqr_pinned_cases():
    """(key, A, B, Q, R) of test_gpu_parity.test_lqr_sweep_matches_reference, in its order and from its seed."""
    rng = np.random.default_rng(21)
    # (37, 5): odd sizes on the tensor-core path (every tile ragged, no vector loads); (40, 6): partial 16 x 40 tiles
    for nX, nU, K, R_, per_step in ((4, 1, 60, 3, False), (80, 18, 25, 2, True), (7, 3, 40, 5, True),
                                    (37, 5, 12, 2, True), (40, 6, 12, 3, False)):
        A = np.eye(nX)[None, None] + rng.normal(0, 0.3 / np.sqrt(nX), (R_, K, nX, nX))
        B = rng.normal(0, 1.0, (R_, K, nX, nU))
        if per_step:
            Qs = np.stack([np.eye(nX) * (1 + 0.1 * k) for k in range(K + 1)])
            Rs = np.stack([np.eye(nU) * (2 + 0.05 * k) for k in range(K)])
        else:
            M = rng.normal(0, 1, (nX, nX)); Qs = M @ M.T + np.eye(nX)
            Rs = np.eye(nU) * 0.5
        yield "lqr_%d_%d" % (nX, nU), A, B, Qs, Rs


def lq_pinned_cases():
    """(key, A, B, q, r, Q, S, R, per_rollout) of test_gpu_parity.test_lq_sweep_matches_reference, in its order and
    from its seed; the cost arrays carry a rollout axis only when per_rollout."""
    rng = np.random.default_rng(22)
    for nX, nU, K, R_, per_rollout, with_s in ((4, 1, 50, 3, False, True), (80, 18, 20, 2, True, True),
                                               (7, 3, 30, 4, True, False), (5, 2, 10, 1, False, False),
                                               (37, 5, 10, 2, True, True)):
        A = np.eye(nX)[None, None] + rng.normal(0, 0.3 / np.sqrt(nX), (R_, K, nX, nX))
        B = rng.normal(0, 1.0, (R_, K, nX, nU))
        nc = R_ if per_rollout else 1
        Qs = np.stack([np.stack([np.eye(nX) * (1 + 0.1 * k + 0.3 * c) for k in range(K + 1)]) for c in range(nc)])
        Rs = np.stack([np.stack([np.eye(nU) * (2 + 0.05 * k + 0.2 * c) for k in range(K)]) for c in range(nc)])
        Ss = rng.normal(0, 0.05, (nc, K, nX, nU)) if with_s else None
        q = rng.normal(0, 1, (nc, K + 1, nX)); r = rng.normal(0, 1, (nc, K, nU))
        sq = (lambda x: x) if per_rollout else (lambda x: None if x is None else x[0])
        yield "lq_%d_%d" % (nX, nU), A, B, sq(q), sq(r), sq(Qs), sq(Ss), sq(Rs), per_rollout


# observed: 1.2e-14 (at 80 / 18); the pins are fp64 results of a different summation order
BOUND = 1e-12


def _pin(key):
    with np.load(G.EXPECTED + "/" + key + ".npz") as f:
        return {k: f[k] for k in f.files}


@pytest.mark.parametrize("case", range(5))
def test_reference_reproduces_the_lqr_pins(case):
    key, A, B, Q, R = list(lqr_pinned_cases())[case]
    want = _pin(key)
    for i in range(A.shape[0]):
        K, _, P, _ = lqref.solve_tv_lq_ld(A[i], B[i], Q, R)
        for name, got in (("K", K), ("P", P)):
            e = G.relerr(got.astype(float), want[name][i])
            assert e <= BOUND, "%s %s rollout %d: relerr %.2e" % (key, name, i, e)


@pytest.mark.parametrize("case", range(5))
def test_reference_reproduces_the_lq_pins(case):
    key, A, B, q, r, Q, S, R, per = list(lq_pinned_cases())[case]
    want = _pin(key)
    pick = (lambda x, i: None if x is None else x[i]) if per else (lambda x, i: x)
    for i in range(A.shape[0]):
        K, C, P, b = lqref.solve_tv_lq_ld(A[i], B[i], pick(Q, i), pick(R, i), S=pick(S, i), q=pick(q, i), r=pick(r, i))
        for name, got in (("K", K), ("C", C), ("P", P), ("b", b)):
            e = G.relerr(got.astype(float), want[name][i])
            assert e <= BOUND, "%s %s rollout %d: relerr %.2e" % (key, name, i, e)


def test_batched_fp64_helper_agrees_with_the_long_double_reference():
    """solve_tv_lq_f64 (the whole-batch check of the GPU tests) on the per-rollout-cost pin case with S."""
    key, A, B, q, r, Q, S, R, per = list(lq_pinned_cases())[4]
    assert per and S is not None
    K, C, P, b = lqref.solve_tv_lq_f64(A, B, Q, R, S=S, q=q, r=r)
    for i in range(A.shape[0]):
        want = lqref.solve_tv_lq_ld(A[i], B[i], Q[i], R[i], S=S[i], q=q[i], r=r[i])
        for name, got, w in zip("KCPb", (K, C, P, b), want):
            assert G.relerr(got[i], w.astype(float)) <= BOUND, (key, name, i)


def test_sweep_references_match_their_recurrences():
    """tangent_ld / adjoint_ld against the plain fp64 loops of the existing sweep tests (test_gpu_sweeps.py), with
    and without the optional arrays."""
    rng = np.random.default_rng(3)
    n, nX, nU = 9, 6, 2
    A = 0.3 * rng.normal(size=(n, nX, nX)); B = rng.normal(size=(n, nX, nU)); K = 0.2 * rng.normal(size=(n, nU, nX))
    bdX, bdU, x0 = rng.normal(size=(n + 1, nX)), rng.normal(size=(n, nU)), rng.normal(size=nX)
    l_dx, l_du, m = rng.normal(size=(n, nX)), rng.normal(size=(n, nU)), rng.normal(size=nX)
    for bx, bu, x in ((bdX, bdU, x0), (bdX, bdU, None), (None, bdU, None), (None, None, x0)):
        dX, dU = np.zeros((n + 1, nX)), np.zeros((n, nU))
        dX[0] = x if x is not None else bx[0] if bx is not None else 0
        for k in range(n):
            dU[k] = (0 if bu is None else bu[k]) - K[k] @ (dX[k] - (0 if bx is None else bx[k]))
            dX[k + 1] = A[k] @ dX[k] + B[k] @ dU[k]
        got = lqref.tangent_ld(A, B, K, bx, bu, x)
        G.assert_close(got[0].astype(float), dX, "dX", rtol=1e-13)
        G.assert_close(got[1].astype(float), dU, "dU", rtol=1e-13)
    for Kf, lx, lu in ((K, l_dx, l_du), (None, l_dx, l_du), (K, None, l_du), (K, l_dx, None)):
        z = np.zeros((n + 1, nX)); z[n] = m
        for k in reversed(range(n)):
            z[k] = (0 if lx is None else lx[k]) + A[k].T @ z[k + 1]
            if Kf is not None:
                z[k] -= Kf[k].T @ ((0 if lu is None else lu[k]) + B[k].T @ z[k + 1])
        G.assert_close(lqref.adjoint_ld(A, m, B, Kf, lx, lu).astype(float), z, "z", rtol=1e-13)
