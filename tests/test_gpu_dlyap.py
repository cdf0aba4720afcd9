"""Closed-loop cost and stability of stationary gains on the device (dlyap_kernel behind trepb_dlyap_batch*,
lib.solve_closed_loop and DSystem.evaluate_stationary_controller):

- against scipy.linalg.solve_discrete_lyapunov(A_c^T, Q_c) from 1x1 to the largest shapes the DARE admits, nU > nX
  included, Q / R / S shared and per model, with and without S; a long-double residual; cost = x0^T P x0;
- the stability verdict against numpy.linalg.eigvals, Q_c = 0 on the unstable direction included, and unstable pairs
  every 97th in grid-stride batches leaving their neighbours' bits alone;
- the Lyapunov P of a model's own DARE gain equals the DARE's P;
- bit identity: P symmetric, alone against in a batch, host entry against _dev on a stream, index cross-evaluation
  against the same pairs laid out;
- pend-on-cart upright under 64 models against closed-loop rollouts, and the marionette."""
import numpy as np
import pytest
import scipy.linalg as sla

from test_gpu_dare import dare_smem_bytes, limit_shapes, problem, rtol_for

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


def dlyap_smem_bytes(n, m):
    """Dynamic shared memory dlyap_launch asks for (dlyap_layout, trepb_dlyap.cuh)."""
    ld = (n + 1) | 1
    nw = min(16, max(2, (n * n + 255) // 256))
    blk = n * ld
    return 8 * (3 * blk + max(blk, m * n) + 3 * nw)


# ---- problems and references ---------------------------------------------------------------------------------------

def _spd(rng, shape, n):
    M = rng.normal(size=shape + (n, n))
    return M @ np.swapaxes(M, -1, -2) / n + np.eye(n)


def with_radius(M, rho):
    """M scaled to spectral radius rho."""
    r = np.max(np.abs(np.linalg.eigvals(M)), axis=-1)
    return M * (rho / r)[..., None, None]


def closed_loop_problem(rng, N, nX, nU, per=False, cross=False, rho=0.9):
    """N models whose closed loop under the gain K has spectral radius rho: A = A_c + B K with A_c random at radius
    rho, B and K dense; SPD Q and R (one per model when per), a small cross term S."""
    Ac = with_radius(rng.normal(size=(N, nX, nX)), rho)
    B = rng.normal(size=(N, nX, nU))
    K = rng.normal(0, 1.0 / np.sqrt(nX + nU), (N, nU, nX))
    A = Ac + B @ K
    lead = (N,) if per else ()
    Q, R = _spd(rng, lead, nX), _spd(rng, lead, nU)
    S = rng.normal(0, 0.1 / np.sqrt(nX), lead + (nX, nU)) if cross else None
    return A, B, K, Q, R, S


def pick(x, i, per):
    return None if x is None else (x[i] if per else x)


def closed_loop(A, B, K, Q, R, S, dt=float):
    A, B, K, Q, R = (np.array(x, dtype=dt) for x in (A, B, K, Q, R))
    Ac = A - B @ K
    Qc = (Q + Q.T) / 2 + K.T @ ((R + R.T) / 2) @ K
    if S is not None:
        S = np.array(S, dtype=dt)
        Qc = Qc - S @ K - K.T @ S.T
    return Ac, Qc


def check_against_scipy(A, B, K, Q, R, S, P, what, rtol=1e-10):
    Ac, Qc = closed_loop(A, B, K, Q, R, S)
    Pw = sla.solve_discrete_lyapunov(Ac.T, Qc)
    e = np.max(np.abs(P - Pw)) / np.max(np.abs(Pw))
    assert e <= rtol, (what, e)
    # the residual in extended precision, against the size of its terms
    Ac, Qc = closed_loop(A, B, K, Q, R, S, LD)
    Pl = np.array(P, dtype=LD)
    apa = Ac.T @ Pl @ Ac
    res = apa - Pl + Qc
    terms = np.sqrt(np.sum(apa * apa) + np.sum(Pl * Pl) + np.sum(Qc * Qc))
    assert float(np.sqrt(np.sum(res * res)) / terms) <= 1e-12, what


def run(lib, A, B, K, Q, R, S=None, gain_index=None, model_index=None, x0=None, W=None, **kw):
    M, nX, nU = B.shape
    G = K.shape[0]
    n = len(gain_index) if gain_index is not None else len(model_index) if model_index is not None else M
    P, cost = np.full((n, nX, nX), np.nan), np.full(n, np.nan)
    st, it = np.full(n, 7, np.int32), np.zeros(n, np.int32)
    has_cost = x0 is not None or W is not None
    lib.dlyap_raw(False, 0, n, G, M, nX, nU, A, B, K, Q, R, st, S=S, gain_index=gain_index, model_index=model_index,
                  x0=x0, W=W, P=P, cost=cost if has_cost else None, iterations=it, q_per_model=Q.ndim == 3,
                  r_per_model=R.ndim == 3, s_per_model=S is not None and S.ndim == 3,
                  x0_per_pair=x0 is not None and x0.ndim == 2, **kw)
    return P, cost, st, it


def quad_ld(x, P):
    """x^T P x in long double, and the sum of the magnitudes of its terms."""
    x, P = np.array(x, dtype=LD), np.array(P, dtype=LD)
    return float(x @ P @ x), float(np.abs(x) @ np.abs(P) @ np.abs(x))


# ---- against scipy --------------------------------------------------------------------------------------------------

SHAPES = [(1, 1), (2, 1), (4, 1), (7, 3), (3, 5), (32, 31), (80, 18), "nX_at_nU1", "nU_at_nX80", "nU_at_nX1"]


@pytest.mark.parametrize("shape", SHAPES, ids=[s if isinstance(s, str) else "%dx%d" % s for s in SHAPES])
@pytest.mark.parametrize("per,cross", [(False, False), (True, False), (False, True), (True, True)],
                         ids=["shared", "per_model", "shared_S", "per_model_S"])
def test_against_scipy(lib, device, shape, per, cross):
    nX, nU = limit_shapes(device["optin"])[shape] if isinstance(shape, str) else shape
    rng = np.random.default_rng(2000 * nX + nU + 7 * per + 3 * cross)
    N = 3
    A, B, K, Q, R, S = closed_loop_problem(rng, N, nX, nU, per, cross)
    x0 = rng.normal(size=(N, nX))
    P, cost, st, it = run(lib, A, B, K, Q, R, S, x0=x0)
    assert np.all(st == lib.DLYAP_STABLE), st
    assert np.all((it >= 1) & (it < 64)), it
    for i in range(N):
        check_against_scipy(A[i], B[i], K[i], pick(Q, i, per), pick(R, i, per), pick(S, i, per), P[i], (nX, nU, i))
        assert np.array_equal(P[i], P[i].T)
        want, scale = quad_ld(x0[i], P[i])
        assert abs(cost[i] - want) <= 1e-12 * scale, (i, cost[i], want)
    # a shared x0 and a weight W: trace(P W)
    W = _spd(rng, (), nX)
    P2, c2, st2, _ = run(lib, A, B, K, Q, R, S, x0=x0[0])
    assert np.all(st2 == 0) and P2.tobytes() == P.tobytes()
    for i in range(N):
        want, scale = quad_ld(x0[0], P[i])
        assert abs(c2[i] - want) <= 1e-12 * scale
    _, c3, _, _ = run(lib, A, B, K, Q, R, S, W=W)
    want = np.einsum("pij,ji->p", P.astype(LD), W.astype(LD))
    assert np.all(np.abs(c3 - want.astype(float)) <= 1e-12 * np.einsum("pij,ji->p", np.abs(P), np.abs(W)))


@pytest.mark.parametrize("nX,nU", [(2, 9), (10, 20), (30, 40), (61, 64)])
def test_more_inputs_than_a_block_row_holds_after_either_doubling_parity(lib, nX, nU):
    """nU nX > nX ((nX + 1) | 1): R K is larger than one n x ld block.  The F / T blocks swap after every squaring, so
    the residual must find the large block after an odd doubling count as after an even one."""
    rng = np.random.default_rng(100 * nX + nU)
    radii = [0.3, 0.5, 0.7, 0.8, 0.9, 0.95, 0.98]
    parities = set()
    for rho in radii:
        A, B, K, Q, R, S = closed_loop_problem(rng, 2, nX, nU, per=True, cross=True, rho=rho)
        x0 = rng.normal(size=(2, nX))
        P, cost, st, it = run(lib, A, B, K, Q, R, S, x0=x0)
        assert np.all(st == lib.DLYAP_STABLE), (rho, st, it)
        parities |= set((it % 2).tolist())
        for i in range(2):
            check_against_scipy(A[i], B[i], K[i], Q[i], R[i], S[i], P[i], (nX, nU, rho, i))
            want, scale = quad_ld(x0[i], P[i])
            assert abs(cost[i] - want) <= 1e-12 * scale
    assert parities == {0, 1}, parities


def test_every_shape_the_dare_admits_is_admitted(lib, device):
    optin = device["optin"]
    for n in range(1, 100):
        for m in range(1, 200):
            if dare_smem_bytes(n, m) <= optin:
                assert dlyap_smem_bytes(n, m) <= optin, (n, m)


def test_one_past_the_limit_is_refused(lib, device):
    optin = device["optin"]
    n = max(k for k in range(1, 400) if dlyap_smem_bytes(k, 1) <= optin) + 1
    assert n > limit_shapes(optin)["nX_at_nU1"][0]
    A, B, K = np.zeros((1, n, n)), np.zeros((1, n, 1)), np.zeros((1, 1, n))
    st = np.full(1, 7, np.int32)
    with pytest.raises(lib.TrepbError) as e:
        lib.dlyap_raw(False, 0, 1, 1, 1, n, 1, A, B, K, np.eye(n), np.eye(1), st)
    assert e.value.code == 4 and "too large for the shared-memory Lyapunov solve" in str(e.value)
    assert "%d bytes of shared memory needed, %d per block" % (dlyap_smem_bytes(n, 1), optin) in str(e.value)
    assert st[0] == 7


def test_solve_closed_loop_single_and_errors(lib):
    rng = np.random.default_rng(5)
    A, B, K, Q, R, S = closed_loop_problem(rng, 1, 5, 2, cross=True)
    x0 = rng.normal(size=5)
    P, cost, st, it = lib.solve_closed_loop(A[0], B[0], K[0], Q, R, S=S, x0=x0)
    assert st == 0 and it >= 1 and P.shape == (5, 5)
    check_against_scipy(A[0], B[0], K[0], Q, R, S, P, "single")
    assert abs(cost - quad_ld(x0, P)[0]) <= 1e-12 * quad_ld(x0, P)[1]
    with pytest.raises(lib.TrepbError, match="not converged"):
        lib.solve_closed_loop(A[0], B[0], K[0], Q, R, max_iterations=1)
    Au = A[0] + 2.0 * np.eye(5)                 # rho(A_c) = 2.9
    with pytest.raises(lib.TrepbError, match="non-finite"):
        lib.solve_closed_loop(Au, B[0], K[0], Q, R)
    # a batch reports and does not raise; the cost of an unstable pair is +inf
    P, cost, st, it = lib.solve_closed_loop(Au[None], B, K, Q, R, x0=x0)
    assert st.tolist() == [lib.DLYAP_NONFINITE] and cost[0] == np.inf


# ---- the stability verdict ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("nX,nU", [(1, 1), (4, 1), (12, 3), (40, 7)])
def test_the_verdict_follows_the_spectral_radius(lib, nX, nU):
    rng = np.random.default_rng(31 * nX + nU)
    radii = [0.2, 0.9, 0.99, 0.999, 1.001, 1.01, 1.1, 2.0]
    N = len(radii)
    _, B, K, Q, R, _ = closed_loop_problem(rng, N, nX, nU)
    Ac = np.stack([with_radius(rng.normal(size=(nX, nX)), r) for r in radii])
    A = Ac + B @ K
    rho = np.max(np.abs(np.linalg.eigvals(A - B @ K)), axis=-1)
    P, cost, st, it = run(lib, A, B, K, Q, R, x0=np.ones(nX))
    stable = rho <= 0.999 * (1 + 1e-12)
    assert np.all(st[stable] == lib.DLYAP_STABLE), (rho, st)
    assert np.all(st[rho >= 1.001 * (1 - 1e-12)] != lib.DLYAP_STABLE), (rho, st)
    assert np.all(np.isfinite(cost[stable])) and np.all(cost[~stable] == np.inf)


@pytest.mark.parametrize("rho", [1.001, 1.01, 1.5, 1.0])
def test_an_unstable_direction_the_cost_does_not_see(lib, rho):
    """Q_c = 0 on the unstable mode: P alone converges (to the cost of the stable part), the test on F does not."""
    n = 5
    rng = np.random.default_rng(int(rho * 1000))
    Ac = np.zeros((n, n))
    Ac[0, 0] = rho
    Ac[1:, 1:] = with_radius(rng.normal(size=(n - 1, n - 1)), 0.5)
    Ac[1:, 0] = 0.0                              # the unstable mode does not feed the observed ones
    Ac[0, 1:] = rng.normal(size=n - 1)
    Q = np.diag([0.0] + [1.0] * (n - 1))
    B, K = np.zeros((1, n, 1)), np.zeros((1, 1, n))
    P, cost, st, it = run(lib, Ac[None], B, K, Q, np.eye(1), x0=np.ones(n))
    assert st[0] in (lib.DLYAP_NOT_CONVERGED, lib.DLYAP_NONFINITE), st
    assert cost[0] == np.inf
    # the stable part alone is certified
    _, _, st2, _ = run(lib, Ac[None, 1:, 1:], B[:, 1:], K[:, :, 1:], Q[1:, 1:], np.eye(1))
    assert st2[0] == lib.DLYAP_STABLE


@pytest.mark.parametrize("nX,nU,N", [(80, 18, None), (4, 1, 10000)], ids=["80x18_2SMs+3", "4x1_10000"])
def test_unstable_pairs_leave_the_others_alone(lib, device, nX, nU, N):
    N = N or 2 * device["sms"] + 3
    rng = np.random.default_rng(nX + N)
    A, B, K, Q, R, S = closed_loop_problem(rng, N, nX, nU, per=True, cross=True)
    x0 = rng.normal(size=(N, nX))
    P0, c0, s0, i0 = run(lib, A, B, K, Q, R, S, x0=x0)
    assert np.all(s0 == 0)
    bad = np.arange(0, N, 97)
    Au = A.copy()
    Au[bad] += 2.0 * np.eye(nX)                 # |lambda + 2| >= 2 - 0.9: rho(A_c) >= 1.1
    rho = np.max(np.abs(np.linalg.eigvals(Au[bad] - B[bad] @ K[bad])), axis=-1)
    assert np.all(rho > 1.001)
    P1, c1, s1, i1 = run(lib, Au, B, K, Q, R, S, x0=x0)
    assert np.all(s1[bad] != 0) and np.all(c1[bad] == np.inf)
    good = np.setdiff1d(np.arange(N), bad)
    assert np.all(s1[good] == 0)
    assert P1[good].tobytes() == P0[good].tobytes() and c1[good].tobytes() == c0[good].tobytes()
    assert np.array_equal(i1[good], i0[good])
    for i in rng.choice(good, 4, replace=False):
        check_against_scipy(A[i], B[i], K[i], Q[i], R[i], S[i], P0[i], i)


@pytest.mark.parametrize("nX,nU", [(4, 1), (12, 3)])
def test_a_bad_index_on_the_dev_entry_is_a_status(lib, nX, nU):
    import torch
    rng = np.random.default_rng(17)
    G, M = 3, 4
    A, B, _, Q, R, _ = closed_loop_problem(rng, M, nX, nU)
    K = rng.normal(0, 0.01, (G, nU, nX))
    gi = np.array([0, 1, 2, 3, 0, -1], np.int32)      # gain 3 and gain -1 do not exist
    mi = np.array([0, 1, 2, 3, 4, 0], np.int32)       # nor does model 4
    t = lambda x: torch.tensor(x, device="cuda")
    st = torch.full((6,), 7, dtype=torch.int32, device="cuda")
    cost = torch.zeros(6, dtype=torch.float64, device="cuda")
    lib.dlyap_raw(True, 0, 6, G, M, nX, nU, t(A), t(B), t(K), t(Q), t(R), st, gain_index=t(gi), model_index=t(mi),
                  W=t(np.eye(nX)), cost=cost)
    torch.cuda.synchronize()
    st, cost = st.cpu().numpy(), cost.cpu().numpy()
    assert st[3:].tolist() == [lib.DLYAP_BAD_INDEX] * 3 and np.all(cost[3:] == np.inf)
    _, c, s, _ = run(lib, A, B, K, Q, R, gain_index=gi[:3], model_index=mi[:3], W=np.eye(nX))
    assert st[:3].tolist() == s.tolist() and cost[:3].tobytes() == c.tobytes()


# ---- the DARE's P is the Lyapunov P of its own gain -------------------------------------------------------------

@pytest.mark.parametrize("nX,nU", [(4, 1), (7, 3), (3, 5), (12, 3), (32, 31), (80, 18)])
@pytest.mark.parametrize("cross", [False, True], ids=["noS", "S"])
def test_the_dare_gain_gives_the_dare_cost(lib, nX, nU, cross):
    rng = np.random.default_rng(4000 + 10 * nX + nU + cross)
    N = 4
    A, B, Q, R, S = problem(rng, N, nX, nU, per=True, cross=cross)
    K, P, st, _ = lib.solve_dare(A, B, Q, R, S=S)
    assert np.all(st == 0)
    Pl, _, sl, _ = lib.solve_closed_loop(A, B, K, Q, R, S=S)
    assert np.all(sl == lib.DLYAP_STABLE), sl
    for i in range(N):
        rt = rtol_for(A[i], B[i], Q[i], R[i], K[i], P[i])
        e = np.max(np.abs(Pl[i] - P[i])) / np.max(np.abs(P[i]))
        assert e <= rt, (i, e, rt)


# ---- bit identity ---------------------------------------------------------------------------------------------------

def test_alone_against_in_a_batch_of_1000(lib):
    rng = np.random.default_rng(1000)
    N, nX, nU = 1000, 9, 4
    A, B, K, Q, R, S = closed_loop_problem(rng, N, nX, nU, per=True, cross=True)
    x0 = rng.normal(size=(N, nX))
    P, c, st, it = run(lib, A, B, K, Q, R, S, x0=x0)
    assert np.all(st == 0)
    for i in rng.choice(N, 12, replace=False):
        sl = slice(i, i + 1)
        p1, c1, s1, i1 = run(lib, A[sl], B[sl], K[sl], Q[sl], R[sl], S[sl], x0=x0[sl])
        assert s1[0] == 0 and i1[0] == it[i]
        assert p1[0].tobytes() == P[i].tobytes() and c1[0].tobytes() == c[i].tobytes(), i


def test_dev_entry_on_a_stream_gives_the_host_bits(lib):
    import torch
    rng = np.random.default_rng(12)
    G, M, nX, nU = 5, 7, 12, 3
    A, B, _, Q, R, S = closed_loop_problem(rng, M, nX, nU, per=True, cross=True)
    K = rng.normal(0, 0.02, (G, nU, nX))
    gi, mi = np.repeat(np.arange(G), M).astype(np.int32), np.tile(np.arange(M), G).astype(np.int32)
    x0 = rng.normal(size=(G * M, nX))
    P, c, st, it = run(lib, A, B, K, Q, R, S, gain_index=gi, model_index=mi, x0=x0)
    t = lambda x: torch.tensor(x, device="cuda")
    n = G * M
    dP = torch.zeros((n, nX, nX), dtype=torch.float64, device="cuda")
    dc = torch.zeros(n, dtype=torch.float64, device="cuda")
    dst, dit = torch.zeros(n, dtype=torch.int32, device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        args = [t(x) for x in (A, B, K, Q, R, S, gi, mi, x0)]
        lib.dlyap_raw(True, 0, n, G, M, nX, nU, *args[:5], dst, S=args[5], gain_index=args[6], model_index=args[7],
                      x0=args[8], P=dP, cost=dc, iterations=dit, q_per_model=True, r_per_model=True,
                      s_per_model=True, x0_per_pair=True, stream=s.cuda_stream)
    s.synchronize()
    assert np.array_equal(dst.cpu().numpy(), st) and np.array_equal(dit.cpu().numpy(), it)
    assert dP.cpu().numpy().tobytes() == P.tobytes() and dc.cpu().numpy().tobytes() == c.tobytes()


def test_index_cross_evaluation_against_the_pairs_laid_out(lib):
    rng = np.random.default_rng(13)
    G, M, nX, nU = 6, 9, 8, 2
    A, B, _, Q, R, S = closed_loop_problem(rng, M, nX, nU, per=True, cross=True)
    K = rng.normal(0, 0.05, (G, nU, nX))
    gi, mi = np.repeat(np.arange(G), M).astype(np.int32), np.tile(np.arange(M), G).astype(np.int32)
    P, c, st, it = lib.solve_closed_loop(A, B, K, Q, R, S=S, x0=np.ones(nX), gain_index=gi, model_index=mi)
    assert np.any(st == 0)
    P2, c2, st2, it2 = lib.solve_closed_loop(A[mi], B[mi], K[gi], Q[mi], R[mi], S=S[mi], x0=np.ones(nX))
    assert np.array_equal(st, st2) and np.array_equal(it, it2)
    ok = st == 0
    assert P[ok].tobytes() == P2[ok].tobytes() and c.tobytes() == c2.tobytes()
    # one index alone: the other side is the identity
    P3, c3, st3, _ = lib.solve_closed_loop(A, B, K[:1], Q, R, S=S, x0=np.ones(nX), gain_index=np.zeros(M))
    assert np.array_equal(st3, st[:M]) and c3.tobytes() == c[:M].tobytes()


# ---- end to end -------------------------------------------------------------------------------------------------------

def test_pend_on_cart_nominal_gain_under_64_models(lib):
    """The upright cart-pole's nominal LQR gain under 64 pendulum masses and lengths, some of which it does not
    stabilize: each verdict agrees with the eigenvalues and with a 2000-step closed-loop rollout."""
    import golden_util as G
    from trep_b200 import discopt, midpointvi as MV
    from trep_b200.midpointvi import ConvergenceError
    d = G.desc("pend_on_cart1")
    refs = [d.param_ref("frame_mass", 3, 0), d.param_ref("frame_value", 3)]   # pendulum mass and length
    masses, lengths = [0.5, 1.0, 2.0, 4.0], np.geomspace(0.05, 4.0, 16)
    vals = np.array([(m, -l) for m in masses for l in lengths])
    M = len(vals)
    Kn = 2000
    t = np.arange(Kn + 1) * 0.01
    xk, uk = np.array([0.0, np.pi, 0.0, 0.0]), np.zeros(1)
    Q, Rw = np.diag([100.0, 100.0, 1.0, 1.0]), np.array([[0.01]])
    Knom, Pnom = discopt.DSystem(MV.MidpointVI(d), t).calc_stationary_controller(xk, uk, Q, Rw)
    ds = discopt.DSystem(MV.MidpointVI(d), t)
    ds.set_parameters(refs, vals)
    x0 = np.array([1e-3, 1e-3, 0.0, 0.0])
    cost, st, P = ds.evaluate_stationary_controller(xk, uk, Knom, Q, Rw, x0=x0, return_P=True)
    assert cost.shape == (M,) and st.shape == (M,) and P.shape == (M, 4, 4)
    A, B = ds.linearize(np.tile(xk, (M, 1)), np.tile(uk, (M, 1)), np.full(M, 0.0), np.full(M, 0.01),
                        X_hint=np.tile(xk, (M, 1)))
    rho = np.max(np.abs(np.linalg.eigvals(A - B @ Knom)), axis=-1)
    assert np.all(st[rho <= 0.999] == lib.DLYAP_STABLE), (rho, st)
    assert np.all(st[rho >= 1.001] != lib.DLYAP_STABLE), (rho, st)
    ok = st == 0
    assert np.all(np.isfinite(cost[ok])) and np.all(cost[~ok] == np.inf)
    for r in np.flatnonzero(ok):
        check_against_scipy(A[r], B[r], Knom, Q, Rw, None, P[r], r, rtol=1e-9)
    # rollouts, away from the unit circle (where 2000 steps cannot tell)
    clear = np.abs(rho - 1.0) >= 0.002
    assert np.sum(clear & ok) >= 8 and np.sum(clear & ~ok) >= 8, rho
    bX = np.tile(xk, (M, Kn + 1, 1))
    bX[:, 0] += x0
    try:
        X = ds.project(bX, np.zeros((M, Kn, 1)), np.repeat(Knom[None], Kn, axis=0)).X
        failed = np.zeros(M, bool)
    except ConvergenceError:
        X, failed = ds.last_project["X"], ds.last_project["status"] != 0
    e0 = np.linalg.norm(x0)
    e1 = np.linalg.norm(X[:, -1] - xk, axis=1)
    returns = ~failed & (e1 < 0.5 * e0)
    diverges = failed | ~np.isfinite(e1) | (e1 > 5 * e0)
    assert np.all(returns[clear & ok]), (rho[clear & ok], e1[clear & ok] / e0)
    assert np.all(diverges[clear & ~ok]), (rho[clear & ~ok], e1[clear & ~ok] / e0)
    # the cross-evaluation of G gains holds this one's row, bit for bit
    cost2, st2 = ds.evaluate_stationary_controller(xk, uk, np.stack([Knom, 0.5 * Knom]), Q, Rw, x0=x0)
    assert cost2.shape == (2, M) and np.array_equal(st2[0], st) and cost2[0].tobytes() == cost.tobytes()


def test_pend_on_cart_own_dare_gains_under_64_models(lib):
    """Each model's own DARE gain, evaluated per model (cross=False): the Lyapunov P is the DARE's P."""
    import golden_util as G
    from trep_b200 import discopt, midpointvi as MV
    d = G.desc("pend_on_cart1")
    refs = [d.param_ref("frame_mass", 3, 0), d.param_ref("frame_value", 3)]
    rng = np.random.default_rng(64)
    M = 64
    vals = np.stack([rng.uniform(0.5, 2.0, M), -rng.uniform(0.5, 1.5, M)], axis=1)
    ds = discopt.DSystem(MV.MidpointVI(d), np.arange(11) * 0.01)
    ds.set_parameters(refs, vals)
    xk, uk = np.array([0.0, np.pi, 0.0, 0.0]), np.zeros(1)
    Q, Rw = np.diag([100.0, 100.0, 1.0, 1.0]), np.array([[0.01]])
    K, P, A, B = ds.calc_stationary_controller(xk, uk, Q, Rw, return_linearization=True)
    cost, st, Pl = ds.evaluate_stationary_controller(xk, uk, K, Q, Rw, cross=False, return_P=True)
    assert np.all(st == 0) and np.allclose(cost, np.trace(Pl, axis1=1, axis2=2), rtol=1e-14, atol=0)
    for r in range(M):
        rt = rtol_for(A[r], B[r], Q, Rw, K[r], P[r])
        assert np.max(np.abs(Pl[r] - P[r])) / np.max(np.abs(P[r])) <= rt, r
    # the diagonal of the cross-evaluation, bit for bit
    cc, sc = ds.evaluate_stationary_controller(xk, uk, K, Q, Rw)
    assert cc.shape == (M, M) and np.diagonal(cc).tobytes() == cost.tobytes()
    assert np.array_equal(np.diagonal(sc), st)


def test_marionette_at_rest_under_its_own_dare_gain(lib):
    from test_gpu_doptimizer import _problem
    from trep_b200 import discopt, midpointvi as MV
    d, t, _, X, U, _ = _problem("puppet", 1, 2, 31)
    ds = discopt.DSystem(MV.MidpointVI(d), t)
    assert ds.varint.sys.cooperative
    nX, nU = ds.nX, ds.nU
    Q, Rw = np.eye(nX), np.eye(nU)
    K, P, A, B = ds.calc_stationary_controller(X[0, 0], U[0, 0], Q, Rw, return_linearization=True)
    cost, st, Pl = ds.evaluate_stationary_controller(X[0, 0], U[0, 0], K, Q, Rw, return_P=True)
    assert int(st) == lib.DLYAP_STABLE and Pl.shape == (nX, nX)
    assert np.array_equal(Pl, Pl.T)
    check_against_scipy(A, B, K, Q, Rw, None, Pl, "marionette", rtol=rtol_for(A, B, Q, Rw, K, P))
    assert np.max(np.abs(Pl - P)) / np.max(np.abs(P)) <= rtol_for(A, B, Q, Rw, K, P)
    assert abs(float(cost) - np.trace(Pl)) <= 1e-13 * abs(np.trace(Pl))
