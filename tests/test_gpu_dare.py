"""The stationary-LQR solve on the device (dare_kernel behind trepb_dare_batch*, lib.solve_dare and
DSystem.calc_stationary_controller) against scipy.linalg.solve_discrete_are and a long-double residual:

- shapes 1x1 to the marionette's 80x18, nU > nX, and the largest shapes the launcher's shared-memory sizing admits;
- Q / R / S shared and per model, with and without the cross term S;
- P symmetric bit for bit, A - B K stable;
- grid-stride batches in which every 97th model is unstabilizable or has a singular R: exactly those report it;
- a model alone gives the bits it gives inside the batch, and the _dev entry point on a non-default stream the bits
  of the host-array one;
- pend-on-cart at the upright equilibrium under 64 models (set_parameters), end to end, and the marionette."""
import numpy as np
import pytest
import scipy.linalg as sla

import lqref

pytestmark = pytest.mark.gpu

LD = np.longdouble


@pytest.fixture(scope="module")
def lib():
    from trep_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


@pytest.fixture(scope="module")
def device():
    import torch
    p = torch.cuda.get_device_properties(0)
    return {"optin": p.shared_memory_per_block_optin, "sms": p.multi_processor_count}


# ---- the launch limits, from dare_layout (trepb_dare.cuh) -----------------------------------------------------------

def dare_smem_bytes(n, m):
    """Dynamic shared memory dare_launch asks for."""
    ld, s = (n + 1) | 1, max(n, m)
    nw = min(16, max(2, (s * s + 255) // 256))
    blk = n * ld
    wk = max(2 * blk, 4 * n * m + m * m)
    return 8 * (2 * blk + wk + nw * n + s + 2 * (2 * n + m) + 2 * nw + 2)


def limit_shapes(optin):
    """The largest supported shapes: nX at nU = 1, nU at nX = 80 and nU at nX = 1."""
    fits = lambda n, m: dare_smem_bytes(n, m) <= optin
    return {"nX_at_nU1": (max(n for n in range(1, 400) if fits(n, 1)), 1),
            "nU_at_nX80": (80, max(m for m in range(1, 400) if fits(80, m))),
            "nU_at_nX1": (1, max(m for m in range(1, 400) if fits(1, m)))}


# ---- problems and references ---------------------------------------------------------------------------------------

def _spd(rng, shape, n):
    M = rng.normal(size=shape + (n, n))
    return M @ np.swapaxes(M, -1, -2) / n + np.eye(n)


def problem(rng, N, nX, nU, per=False, cross=False):
    """N random stabilizable / detectable problems: A of spectral radius about 1.1 (some open-loop unstable modes; 0.5
    when there are fewer than nX / 8 inputs, where a random B reaches the slow modes only with a badly conditioned P),
    B dense, SPD Q and R (one per model when per), a small cross term S."""
    A = rng.normal(0, (1.1 if 8 * nU >= nX else 0.5) / np.sqrt(nX), (N, nX, nX))
    B = rng.normal(size=(N, nX, nU))
    lead = (N,) if per else ()
    Q, R = _spd(rng, lead, nX), _spd(rng, lead, nU)
    S = rng.normal(0, 0.1 / np.sqrt(nX), lead + (nX, nU)) if cross else None
    return A, B, Q, R, S


def pick(x, i, per):
    return None if x is None else (x[i] if per else x)


def scipy_dare(A, B, Q, R, S=None):
    P = sla.solve_discrete_are(A, B, Q, R, s=S)
    P = (P + P.T) / 2
    Kp = B.T @ P @ A + (0 if S is None else S.T)
    return np.linalg.solve(R + B.T @ P @ B, Kp), P


def residual_ld(A, B, Q, R, S, P):
    """||DARE residual of P||_F / ||P||_F in long double."""
    A, B, Q, R, P = (np.array(x, dtype=LD) for x in (A, B, Q, R, P))
    S = np.zeros(B.shape, dtype=LD) if S is None else np.array(S, dtype=LD)
    M = A.T @ P @ B + S
    res = A.T @ P @ A - P - M @ lqref.solve_ld(R + B.T @ P @ B, M.T) + Q
    return float(np.sqrt(np.sum(res * res)) / np.sqrt(np.sum(P * P)))


def rtol_for(A, B, Q, R, K, P):
    """1e-10 for well-conditioned problems, scaled up by the closed loop's conditioning: how close A - B K comes to
    the unit circle, the condition number of R + B^T P B, and how far P outgrows Q (a nearly unreachable unstable
    mode)."""
    rho = np.max(np.abs(np.linalg.eigvals(A - B @ K)))
    kappa = np.linalg.cond(R + B.T @ P @ B) / max(1.0 - rho, 1e-6) * max(1.0, np.linalg.norm(P) / np.linalg.norm(Q))
    return 1e-10 * max(1.0, kappa / 1e3)


def check_against_scipy(A, B, Q, R, S, K, P, what):
    Kw, Pw = scipy_dare(A, B, Q, R, S)
    rt = rtol_for(A, B, Q, R, Kw, Pw)
    eP = np.max(np.abs(P - Pw)) / np.max(np.abs(Pw))
    eK = np.max(np.abs(K - Kw)) / max(np.max(np.abs(Kw)), 1e-300)
    assert eP <= rt and eK <= rt, (what, eP, eK, rt)


def run(lib, A, B, Q, R, S=None, **kw):
    N, nX, nU = B.shape
    K, P = np.full((N, nU, nX), np.nan), np.full((N, nX, nX), np.nan)
    st, it = np.full(N, 7, np.int32), np.zeros(N, np.int32)
    lib.dare_raw(False, 0, N, nX, nU, A, B, Q, R, st, K=K, P=P, S=S, iterations=it, q_per_rollout=Q.ndim == 3,
                 r_per_rollout=R.ndim == 3, s_per_rollout=S is not None and S.ndim == 3, **kw)
    return K, P, st, it


# ---- against scipy --------------------------------------------------------------------------------------------------

SHAPES = [(1, 1), (2, 1), (4, 1), (7, 3), (3, 5), (32, 31), (80, 18), "nX_at_nU1", "nU_at_nX80", "nU_at_nX1"]


@pytest.mark.parametrize("shape", SHAPES, ids=[s if isinstance(s, str) else "%dx%d" % s for s in SHAPES])
@pytest.mark.parametrize("per,cross", [(False, False), (True, False), (False, True), (True, True)],
                         ids=["shared", "per_model", "shared_S", "per_model_S"])
def test_against_scipy(lib, device, shape, per, cross):
    nX, nU = limit_shapes(device["optin"])[shape] if isinstance(shape, str) else shape
    rng = np.random.default_rng(1000 * nX + nU + 7 * per + 3 * cross)
    N = 3
    A, B, Q, R, S = problem(rng, N, nX, nU, per, cross)
    K, P, st, it = run(lib, A, B, Q, R, S)
    assert np.all(st == 0), st
    assert np.all((it >= 1) & (it < 64)), it
    for i in range(N):
        Qi, Ri, Si = pick(Q, i, per), pick(R, i, per), pick(S, i, per)
        check_against_scipy(A[i], B[i], Qi, Ri, Si, K[i], P[i], (nX, nU, i))
        # properties: symmetric bit for bit, a stable closed loop, a small residual in extended precision
        assert np.array_equal(P[i], P[i].T)
        assert np.max(np.abs(np.linalg.eigvals(A[i] - B[i] @ K[i]))) < 1
        assert residual_ld(A[i], B[i], Qi, Ri, Si, P[i]) <= 1e-12, (nX, nU, i)


def test_one_past_the_limits_is_refused(lib, device):
    for name, (nX, nU) in limit_shapes(device["optin"]).items():
        bigger = (nX + 1, nU) if name == "nX_at_nU1" else (nX, nU + 1)
        assert dare_smem_bytes(*bigger) > device["optin"]
        n, m = bigger
        A, B = np.zeros((1, n, n)), np.zeros((1, n, m))
        st = np.full(1, 7, np.int32)
        with pytest.raises(lib.TrepbError) as e:
            lib.dare_raw(False, 0, 1, n, m, A, B, np.eye(n), np.eye(m), st)
        assert e.value.code == 4 and "too large for the shared-memory DARE solve" in str(e.value)
        assert st[0] == 7


def test_solve_dare_single_and_errors(lib):
    rng = np.random.default_rng(3)
    A, B, Q, R, S = problem(rng, 1, 5, 2, cross=True)
    K, P, st, it = lib.solve_dare(A[0], B[0], Q, R, S=S)
    assert st == 0 and it >= 1 and K.shape == (2, 5) and P.shape == (5, 5)
    check_against_scipy(A[0], B[0], Q, R, S, K, P, "single")
    # a tolerance that cannot be met within one doubling step
    with pytest.raises(lib.TrepbError, match="not converged"):
        lib.solve_dare(A[0], B[0], Q, R, max_iterations=1)
    with pytest.raises(lib.TrepbError, match="singular"):
        lib.solve_dare(A[0], B[0], Q, np.zeros((2, 2)))
    # a batch reports and does not raise
    K, P, st, it = lib.solve_dare(A, B, Q, np.zeros((2, 2)))
    assert st.tolist() == [lib.DARE_SINGULAR]


# ---- failing models in a grid-stride batch ----------------------------------------------------------------------------

@pytest.mark.parametrize("nX,nU,N", [(80, 18, None), (4, 1, 10000)], ids=["80x18_2SMs+3", "4x1_10000"])
def test_failing_models_leave_the_others_alone(lib, device, nX, nU, N):
    N = N or 2 * device["sms"] + 3
    rng = np.random.default_rng(nX + N)
    A, B, Q, R, S = problem(rng, N, nX, nU, per=True)
    bad = np.arange(0, N, 97)
    unstab, sing = bad[0::2], bad[1::2]
    for i in unstab:          # an unstable mode (1.5) B cannot reach: no stabilizing solution
        A[i, 0, :] = 0.0
        A[i, 0, 0] = 1.5
        B[i, 0, :] = 0.0
    for i in sing:            # an exactly singular R
        R[i, -1, :] = 0.0
        R[i, :, -1] = 0.0
    K, P, st, it = run(lib, A, B, Q, R)
    assert np.all(st[sing] == lib.DARE_SINGULAR), st[sing]
    assert np.all(st[unstab] != 0), st[unstab]
    good = np.setdiff1d(np.arange(N), bad)
    assert np.all(st[good] == 0)
    for i in good:
        check_against_scipy(A[i], B[i], Q[i], R[i], None, K[i], P[i], i)
    # bit-identity: a sampled model solved alone
    for i in rng.choice(good, 8, replace=False):
        k1, p1, s1, i1 = run(lib, A[i:i + 1], B[i:i + 1], Q[i:i + 1], R[i:i + 1])
        assert s1[0] == 0 and i1[0] == it[i]
        assert k1[0].tobytes() == K[i].tobytes() and p1[0].tobytes() == P[i].tobytes(), i


def test_dev_entry_on_a_stream_gives_the_host_bits(lib):
    import torch
    rng = np.random.default_rng(11)
    N, nX, nU = 37, 12, 3
    A, B, Q, R, S = problem(rng, N, nX, nU, per=True, cross=True)
    K, P, st, it = run(lib, A, B, Q, R, S)
    t = lambda x: torch.tensor(x, device="cuda")
    dA, dB, dQ, dR, dS = (t(x) for x in (A, B, Q, R, S))
    dK, dP = torch.zeros((N, nU, nX), dtype=torch.float64, device="cuda"), torch.zeros((N, nX, nX), dtype=torch.float64, device="cuda")
    dst, dit = torch.zeros(N, dtype=torch.int32, device="cuda"), torch.zeros(N, dtype=torch.int32, device="cuda")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        lib.dare_raw(True, 0, N, nX, nU, dA, dB, dQ, dR, dst, K=dK, P=dP, S=dS, iterations=dit, q_per_rollout=True,
                     r_per_rollout=True, s_per_rollout=True, stream=s.cuda_stream)
    s.synchronize()
    assert np.array_equal(dst.cpu().numpy(), st) and np.array_equal(dit.cpu().numpy(), it)
    assert dK.cpu().numpy().tobytes() == K.tobytes() and dP.cpu().numpy().tobytes() == P.tobytes()
    # K / P may be left out
    st2 = np.zeros(N, np.int32)
    lib.dare_raw(False, 0, N, nX, nU, A, B, Q, R, st2, S=S, q_per_rollout=True, r_per_rollout=True, s_per_rollout=True)
    assert np.array_equal(st2, st)


# ---- end to end -------------------------------------------------------------------------------------------------------

def test_pend_on_cart_upright_under_64_models(lib):
    import golden_util as G
    from trep_b200 import discopt, midpointvi as MV
    d = G.desc("pend_on_cart1")
    refs = [d.param_ref("frame_mass", 3, 0), d.param_ref("frame_value", 3)]   # pendulum mass and length
    rng = np.random.default_rng(64)
    M = 64
    vals = np.stack([rng.uniform(0.5, 2.0, M), -rng.uniform(0.5, 1.5, M)], axis=1)
    Kn = 2000
    t = np.arange(Kn + 1) * 0.01
    ds = discopt.DSystem(MV.MidpointVI(d), t)
    ds.set_parameters(refs, vals)
    xk, uk = np.array([0.0, np.pi, 0.0, 0.0]), np.zeros(1)
    Q, Rw = np.diag([100.0, 100.0, 1.0, 1.0]), np.array([[0.01]])
    K, P, A, B = ds.calc_stationary_controller(xk, uk, Q, Rw, return_linearization=True)
    assert K.shape == (M, 1, 4) and P.shape == (M, 4, 4)
    # the same solve on the downloaded linearizations, bit for bit
    K2, P2, st, _ = lib.solve_dare(A, B, Q, Rw)
    assert np.all(st == 0) and K2.tobytes() == K.tobytes() and P2.tobytes() == P.tobytes()
    for r in range(M):
        check_against_scipy(A[r], B[r], Q, Rw, None, K[r], P[r], r)
        assert np.max(np.abs(np.linalg.eigvals(A[r] - B[r] @ K[r]))) < 1
    # one DSystem per model, bit for bit
    for r in range(M):
        one = discopt.DSystem(MV.MidpointVI(d.with_params(refs, vals[r])), t)
        k1, p1 = one.calc_stationary_controller(xk, uk, Q, Rw)
        assert k1.tobytes() == K[r].tobytes() and p1.tobytes() == P[r].tobytes(), r
    # the closed loop of every model returns to the upright equilibrium from a perturbed state
    bX = np.tile(xk, (M, Kn + 1, 1))
    bX[:, 0] += np.array([0.1, 0.1, 0.0, 0.0])
    bU = np.zeros((M, Kn, 1))
    X, _ = ds.project(bX, bU, np.repeat(K[:, None], Kn, axis=1))
    e0 = np.linalg.norm(X[:, 0] - xk, axis=1)
    e1 = np.linalg.norm(X[:, -1] - xk, axis=1)
    assert np.all(e1 < 1e-2 * e0), e1 / e0


def test_marionette_on_a_cooperative_handle(lib):
    from test_gpu_doptimizer import _problem
    from test_gpu_varied_deriv2 import _refs
    from trep_b200 import discopt, midpointvi as MV
    d, t, _, X, U, _ = _problem("puppet", 1, 2, 31)
    refs = _refs(d)
    vals = np.array([d.param_value(r) for r in refs]) * np.random.default_rng(32).uniform(0.97, 1.03, (2, len(refs)))
    ds = discopt.DSystem(MV.MidpointVI(d), t)
    assert ds.varint.sys.cooperative
    ds.set_parameters(refs, vals)
    nX, nU = ds.nX, ds.nU
    assert (nX, nU) == (80, 18)
    Q, Rw = np.eye(nX), np.eye(nU)
    K, P, A, B = ds.calc_stationary_controller(X[0, 0], U[0, 0], Q, Rw, return_linearization=True)
    for r in range(2):
        check_against_scipy(A[r], B[r], Q, Rw, None, K[r], P[r], r)
        assert np.array_equal(P[r], P[r].T)
