"""Tangent and adjoint sweeps on the device (trepb_tangent_batch*, trepb_adjoint_batch*) and
DSystem.calc_descent_direction, the chain linearize -> LQR -> (adjoint -> deriv2) -> LQ -> tangent sweep.

- The sweeps against DSystem.dproject and the costate recursion of DSystem.calc_newton_model on random
  linearizations, with every optional array NULL in turn and without inputs.
- The sweeps against the long-double recurrences of tests/lqref.py at every branch of sweep_launch: each team width
  (1 to 128 lanes, rows beyond 128 strided), each ring depth (8, 4, 2) with nsteps around it, a last CTA with idle
  teams, and the refusal one state past the shared-memory limit.
- A rollout alone and inside larger batches gives the same bits, in the host-pointer and the _dev forms.
- The open-loop costate of a real system equals the central difference of a tracking cost through DSystem.simulate.
- calc_descent_direction against the composition of the existing calls it replaces, and with per-rollout parameters
  against one DSystem per rollout."""
import numpy as np
import pytest

import golden_util as G
import lqref
from test_gpu_varied_deriv2 import _refs, _traj
from trep_b200 import discopt, lib as L, midpointvi as MV

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    if L.device_count() < 1:
        pytest.skip("needs a CUDA device")
    return L


def linearization(R, K, nX, nU, seed):
    """A [R,K,nX,nX] = 0.99 x an orthogonal matrix (spectral radius 0.99), B [R,K,nX,nU], gains [R,K,nU,nX] small
    enough that A - B K stays near the unit circle over a few hundred steps."""
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.normal(size=(R, K, nX, nX)))
    s = 1.0 / np.sqrt(nX)
    return 0.99 * Q, 0.3 * s * rng.normal(size=(R, K, nX, nU)), 0.1 * s * rng.normal(size=(R, K, nU, nX)), rng


def assert_rollouts_close(a, b, what):
    """|a - b| <= 1e-12 |b| + 1e-14 max|b|, max taken over each rollout."""
    for r in range(b.shape[0]):
        scale = float(np.max(np.abs(b[r])))
        bad = ~(np.abs(a[r] - b[r]) <= 1e-12 * np.abs(b[r]) + 1e-14 * scale)
        assert not np.any(bad), "%s rollout %d: max |a-b| = %.3e (max|b| = %.3e)" % (
            what, r, float(np.max(np.abs(a[r] - b[r]))), scale)


def costate(A, B, K, l_dx, l_du, m_dx):
    """The recursion of DSystem.calc_newton_model (K None: the open-loop costate)."""
    R, n, nX = A.shape[0], A.shape[1], A.shape[2]
    Z = np.zeros((R, n + 1, nX))
    Z[:, n] = m_dx
    for k in reversed(range(n)):
        if K is None:
            Z[:, k] = l_dx[:, k] + np.einsum("rx,rxy->ry", Z[:, k + 1], A[:, k])
        else:
            Acl = A[:, k] - np.einsum("rxu,ruy->rxy", B[:, k], K[:, k])
            Z[:, k] = l_dx[:, k] - np.einsum("ru,rux->rx", l_du[:, k], K[:, k]) + np.einsum("rx,rxy->ry", Z[:, k + 1], Acl)
    return Z


def tangent_from(A, B, K, bdX, bdU, x0):
    """DSystem.dproject's recursion with dX[0] = x0 (bdX[0] when x0 is None)."""
    dX, dU = np.zeros(bdX.shape), np.zeros(bdU.shape)
    dX[:, 0] = bdX[:, 0] if x0 is None else x0
    for k in range(bdX.shape[1] - 1):
        dU[:, k] = bdU[:, k] - np.einsum("rij,rj->ri", K[:, k], dX[:, k] - bdX[:, k])
        dX[:, k + 1] = np.einsum("rij,rj->ri", A[:, k], dX[:, k]) + np.einsum("rij,rj->ri", B[:, k], dU[:, k])
    return dX, dU


SHAPES = [(4, 1), (7, 3), (80, 18)]


@gpu
@pytest.mark.parametrize("nX,nU", SHAPES, ids=["4x1", "7x3", "80x18"])
def test_tangent_sweep_matches_dproject(lib, nX, nU):
    R, K = 3, 200
    A, B, Kf, rng = linearization(R, K, nX, nU, nX)
    bdX, bdU, x0 = rng.normal(size=(R, K + 1, nX)), rng.normal(size=(R, K, nU)), rng.normal(size=(R, nX))
    dproject = lambda bx, bu: discopt.DSystem.dproject(discopt.DSystem, A, B, bx, bu, Kf)
    want = dproject(bdX, bdU)
    got = lib.tangent_sweep(A, B, Kf, bdX, bdU)
    assert_rollouts_close(got[0], want.dX, "dX")
    assert_rollouts_close(got[1], want.dU, "dU")
    # NULL bdX / bdU (zero) and an explicit dX[0]: dproject's loop from dX[0] = x0
    zX, zU = np.zeros_like(bdX), np.zeros_like(bdU)
    for bx_, bu_, x0_ in ((bdX, bdU, x0), (None, bdU, x0), (bdX, None, None), (None, None, x0), (None, bdU, None)):
        want = tangent_from(A, B, Kf, zX if bx_ is None else bx_, zU if bu_ is None else bu_, x0_)
        got = lib.tangent_sweep(A, B, Kf, bx_, bu_, x0=x0_)
        assert_rollouts_close(got[0], want[0], "dX null")
        assert_rollouts_close(got[1], want[1], "dU null")
    # one trajectory without the rollout axis
    got = lib.tangent_sweep(A[0], B[0], Kf[0], bdX[0], bdU[0])
    assert_rollouts_close(got[0][None], dproject(bdX, bdU).dX[:1], "dX single")


@gpu
def test_tangent_sweep_without_inputs(lib):
    R, K, nX = 2, 50, 5
    A, _, _, rng = linearization(R, K, nX, 1, 3)
    B, Kf = np.zeros((R, K, nX, 0)), np.zeros((R, K, 0, nX))
    bdX = rng.normal(size=(R, K + 1, nX))
    want = discopt.DSystem.dproject(discopt.DSystem, A, B, bdX, np.zeros((R, K, 0)), Kf)
    dX, dU = lib.tangent_sweep(A, B, Kf, bdX, None)
    assert dU.shape == (R, K, 0)
    assert_rollouts_close(dX, want.dX, "dX nU=0")


@gpu
@pytest.mark.parametrize("nX,nU", SHAPES, ids=["4x1", "7x3", "80x18"])
def test_adjoint_sweep_matches_the_newton_model_recursion(lib, nX, nU):
    R, K = 3, 200
    A, B, Kf, rng = linearization(R, K, nX, nU, 100 + nX)
    l_dx, l_du, m_dx = rng.normal(size=(R, K, nX)), rng.normal(size=(R, K, nU)), rng.normal(size=(R, nX))
    assert_rollouts_close(lib.adjoint_sweep(A, B, m_dx, l_dx, l_du, K=Kf), costate(A, B, Kf, l_dx, l_du, m_dx), "z")
    assert_rollouts_close(lib.adjoint_sweep(A, B, m_dx, l_dx, l_du), costate(A, B, None, l_dx, l_du, m_dx), "z open")
    zx, zu = np.zeros_like(l_dx), np.zeros_like(l_du)
    assert_rollouts_close(lib.adjoint_sweep(A, B, m_dx, None, l_du, K=Kf), costate(A, B, Kf, zx, l_du, m_dx), "z l_dx")
    assert_rollouts_close(lib.adjoint_sweep(A, B, m_dx, l_dx, None, K=Kf), costate(A, B, Kf, l_dx, zu, m_dx), "z l_du")
    assert_rollouts_close(lib.adjoint_sweep(A, B, m_dx, None, None), costate(A, B, None, zx, zu, m_dx), "z none")
    # without inputs: the open-loop costate
    B0 = np.zeros((R, K, nX, 0))
    assert_rollouts_close(lib.adjoint_sweep(A, B0, m_dx, l_dx), costate(A, B0, None, l_dx, None, m_dx), "z nU=0")


def _dev_sweeps(lib, A, B, Kf, v1, v2, v3):
    """Both sweeps through the _dev entry points; returns (dX, dU, z, z1)."""
    R, K, nX, nU = A.shape[0], A.shape[1], A.shape[2], B.shape[3]
    up = lambda a: lib.DeviceBuffer(0, a.shape).upload(a)
    dA, dB, dK, d1, d2, d3 = up(A), up(B), up(Kf), up(v1), up(v2), up(v3)
    dX, dU = lib.DeviceBuffer(0, (R, K + 1, nX)), lib.DeviceBuffer(0, (R, K, nU))
    z, z1 = lib.DeviceBuffer(0, (R, K + 1, nX)), lib.DeviceBuffer(0, (R, K, nX))
    lib.tangent_raw(True, 0, R, K, nX, nU, dA, dB, dK, dX, dU, bdX=d1, bdU=d2)
    lib.adjoint_raw(True, 0, R, K, nX, nU, dA, dB, d3, z, K=dK, l_dx=lib.DeviceBuffer(0, (R, K, nX)).upload(v1[:, :K]),
                    l_du=d2, z1=z1)
    lib.synchronize(0)
    return dX.download(), dU.download(), z.download(), z1.download()


@gpu
@pytest.mark.parametrize("nX,nU", [(4, 1), (80, 18)], ids=["4x1", "80x18"])
def test_a_rollout_gives_the_same_bits_alone_and_in_a_batch(lib, nX, nU):
    K = 40
    A, B, Kf, rng = linearization(1000, K, nX, nU, 7)
    bdX, bdU, m_dx = rng.normal(size=(1000, K + 1, nX)), rng.normal(size=(1000, K, nU)), rng.normal(size=(1000, nX))
    l_dx = np.ascontiguousarray(bdX[:, :K])
    full_t = lib.tangent_sweep(A, B, Kf, bdX, bdU)
    full_a = lib.adjoint_sweep(A, B, m_dx, l_dx, bdU, K=Kf)
    full_d = _dev_sweeps(lib, A, B, Kf, bdX, bdU, m_dx)
    assert full_d[0].tobytes() == full_t[0].tobytes() and full_d[1].tobytes() == full_t[1].tobytes()
    assert full_d[2].tobytes() == full_a.tobytes()
    assert full_d[3].tobytes() == full_a[:, 1:].tobytes()
    for lo, hi in ((517, 518), (0, 1), (999, 1000), (300, 337)):
        s = slice(lo, hi)
        t = lib.tangent_sweep(A[s], B[s], Kf[s], bdX[s], bdU[s])
        a = lib.adjoint_sweep(A[s], B[s], m_dx[s], l_dx[s], bdU[s], K=Kf[s])
        dv = _dev_sweeps(lib, *(np.ascontiguousarray(x[s]) for x in (A, B, Kf, bdX, bdU, m_dx)))
        for got, want, what in ((t[0], full_t[0], "dX"), (t[1], full_t[1], "dU"), (a, full_a, "z"),
                                (dv[0], full_t[0], "dX dev"), (dv[1], full_t[1], "dU dev"), (dv[2], full_a, "z dev")):
            assert got.tobytes() == want[s].tobytes(), "%s rollouts %d:%d" % (what, lo, hi)


# ---- sweep_launch's branches against the long-double recurrences (tests/lqref.py) ------------------------------

def sweep_stage(nX, nU):
    """Doubles of one staged step (trepb_sweep.cuh): A, B, K in rows padded to an odd length, two vectors."""
    s = nX * (nX | 1) + nX * (nU | 1) + nU * (nX | 1) + nX + nU
    return (s + 1) & ~1


def sweep_geometry(nX, nU, optin):
    """(team, teams per CTA, ring depth) as sweep_launch picks them; depth 0: refused."""
    team = 1
    while team < max(nX, nU) and team < 128:
        team <<= 1
    teams = max(64, team) // team
    stages = 8
    while stages >= 2 and teams * (stages * sweep_stage(nX, nU) + 2 * nX + nU + 2) * 8 > optin:
        stages //= 2
    return team, teams, stages if stages >= 2 else 0


def _optin():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def ring_shape(spec, optin):
    """"ringD": the largest nX (nU = 2) whose ring is D steps deep; "ring_max+1": one past the largest nX that fits."""
    depth = lambda x: sweep_geometry(x, 2, optin)[2]
    if spec == "ring_max+1":
        return max(x for x in range(1, 1024) if depth(x)) + 1, 2
    return max(x for x in range(1, 1024) if depth(x) == int(spec[4:])), 2


# team 1 / 8; 32 -> 64 lanes; 64 -> 128 lanes (one team per CTA); rows beyond 128 strided; each ring depth at its
# largest state (depth 2: the largest state that fits)
SWEEP_SHAPES = [(1, 1), (2, 5), (32, 1), (33, 1), (64, 3), (65, 3), (4, 130), "ring8", "ring4", "ring2"]


def _sweep_cases():
    # nsteps in {1, stages - 1, stages, stages + 1}: the prologue with fewer steps than the ring holds, a full ring,
    # one wrap; resolved at run time (the depth depends on the device's shared memory)
    return [(s, j) for s in SWEEP_SHAPES for j in range(4)]


@gpu
@pytest.mark.parametrize("spec,which", _sweep_cases(),
                         ids=["%s-%s" % (s if isinstance(s, str) else "%dx%d" % s, ("1", "S-1", "S", "S+1")[j])
                              for s, j in _sweep_cases()])
def test_sweeps_match_the_long_double_recurrences_at_every_team_width_and_ring_depth(lib, spec, which):
    """teams x 3 + 1 rollouts (the last CTA has idle teams), every rollout against lqref.tangent_ld / adjoint_ld at
    1e-12, with all optional arrays and with each left out: tangent without bdX / x0 / bdU; adjoint with z1, without
    K (open loop) and without l_dx / l_du.  The last rollout and one inside the batch give the same bits alone."""
    optin = _optin()
    nX, nU = ring_shape(spec, optin) if isinstance(spec, str) else spec
    team, teams, S = sweep_geometry(nX, nU, optin)
    n = (1, S - 1, S, S + 1)[which]
    if which == 1 and n == 1:
        pytest.skip("a ring of 2: stages - 1 = 1 is the nsteps = 1 case")
    R = teams * 3 + 1
    A, B, Kf, rng = linearization(R, n, nX, nU, 1000 * nX + nU + n)
    bdX, bdU, x0 = rng.normal(size=(R, n + 1, nX)), rng.normal(size=(R, n, nU)), rng.normal(size=(R, nX))
    l_dx, l_du, m_dx = rng.normal(size=(R, n, nX)), rng.normal(size=(R, n, nU)), rng.normal(size=(R, nX))
    what = "%dx%d team %d x %d, ring %d, K=%d" % (nX, nU, team, teams, S, n)
    ld = lambda f, *a: np.stack([f(*(None if x is None else x[i] for x in a)).astype(float) for i in range(R)])

    def tangent(s, bx, bu, x):
        sub = lambda v: None if v is None else np.ascontiguousarray(v[s])
        m = len(range(R)[s])
        dX, dU = np.zeros((m, n + 1, nX)), np.zeros((m, n, nU))
        lib.tangent_raw(False, 0, m, n, nX, nU, sub(A), sub(B), sub(Kf), dX, dU, bdX=sub(bx), bdU=sub(bu), x0=sub(x))
        return dX, dU

    def adjoint(s, K, lx, lu):
        sub = lambda v: None if v is None else np.ascontiguousarray(v[s])
        m = len(range(R)[s])
        z, z1 = np.zeros((m, n + 1, nX)), np.zeros((m, n, nX))
        lib.adjoint_raw(False, 0, m, n, nX, nU, sub(A), sub(B), sub(m_dx), z, K=sub(K), l_dx=sub(lx), l_du=sub(lu),
                        z1=z1)
        return z, z1

    full = slice(0, R)
    for bx, bu, x in ((bdX, bdU, x0), (bdX, bdU, None), (None, bdU, None), (None, None, x0)):
        dX, dU = tangent(full, bx, bu, x)
        want = [ld(lambda *a: lqref.tangent_ld(*a)[j], A, B, Kf, bx, bu, x) for j in range(2)]
        tag = "%s tangent bdX %s bdU %s x0 %s" % (what, bx is not None, bu is not None, x is not None)
        assert_rollouts_close(dX, want[0], tag + " dX")
        assert_rollouts_close(dU, want[1], tag + " dU")
    for K, lx, lu in ((Kf, l_dx, l_du), (None, l_dx, l_du), (Kf, None, l_du), (Kf, l_dx, None)):
        z, z1 = adjoint(full, K, lx, lu)
        want = ld(lambda a, m, b, k, x, u: lqref.adjoint_ld(a, m, b, k, x, u), A, m_dx, B, K, lx, lu)
        tag = "%s adjoint K %s l_dx %s l_du %s" % (what, K is not None, lx is not None, lu is not None)
        assert_rollouts_close(z, want, tag + " z")
        assert z1.tobytes() == np.ascontiguousarray(z[:, 1:]).tobytes(), tag + " z1 = z[1:]"
    fX, fU = tangent(full, bdX, bdU, x0)
    fz, fz1 = adjoint(full, Kf, l_dx, l_du)
    for i in sorted({R - 1, R // 2}):
        s = slice(i, i + 1)
        for got, want, name in zip(tangent(s, bdX, bdU, x0) + adjoint(s, Kf, l_dx, l_du), (fX, fU, fz, fz1),
                                   ("dX", "dU", "z", "z1")):
            assert got.tobytes() == want[s].tobytes(), "%s rollout %d alone: %s" % (what, i, name)


@gpu
@pytest.mark.parametrize("spec", [(1, 0), (33, 0), "ring2"], ids=["1x0", "33x0", "ring2x0"])
def test_sweeps_without_inputs_match_the_long_double_recurrences(lib, spec):
    optin = _optin()
    nX = ring_shape(spec, optin)[0] if isinstance(spec, str) else spec[0]
    team, teams, S = sweep_geometry(nX, 0, optin)
    assert S >= 2
    R, n = teams * 3 + 1, S + 1
    A, _, _, rng = linearization(R, n, nX, 1, 9 + nX)
    bdX, l_dx, m_dx = rng.normal(size=(R, n + 1, nX)), rng.normal(size=(R, n, nX)), rng.normal(size=(R, nX))
    dX = np.zeros((R, n + 1, nX))
    lib.tangent_raw(False, 0, R, n, nX, 0, A, None, None, dX, None, bdX=bdX)
    assert_rollouts_close(dX, np.stack([lqref.tangent_ld(A[i], bdX=bdX[i])[0].astype(float) for i in range(R)]),
                          "%dx0 dX" % nX)
    z = np.zeros((R, n + 1, nX))
    lib.adjoint_raw(False, 0, R, n, nX, 0, A, None, m_dx, z, l_dx=l_dx)
    assert_rollouts_close(z, np.stack([lqref.adjoint_ld(A[i], m_dx[i], l_dx=l_dx[i]).astype(float) for i in range(R)]),
                          "%dx0 z" % nX)


@gpu
def test_sweep_refuses_the_state_one_past_the_shared_memory_limit(lib):
    nX, nU = ring_shape("ring_max+1", _optin())
    A, B, Kf = np.zeros((1, 1, nX, nX)), np.zeros((1, 1, nX, nU)), np.zeros((1, 1, nU, nX))
    dX, dU, z = np.full((1, 2, nX), 0.5), np.full((1, 1, nU), 0.5), np.full((1, 2, nX), 0.5)
    for call in (lambda: lib.tangent_raw(False, 0, 1, 1, nX, nU, A, B, Kf, dX, dU),
                 lambda: lib.adjoint_raw(False, 0, 1, 1, nX, nU, A, B, np.zeros((1, nX)), z, K=Kf)):
        with pytest.raises(lib.TrepbError) as e:
            call()
        assert e.value.code == 4 and "state dimension too large for the shared-memory sweep" in str(e.value)
    assert np.all(dX == 0.5) and np.all(dU == 0.5) and np.all(z == 0.5)


def _dsys(d, t, params=None, **kw):
    ds = discopt.DSystem(MV.MidpointVI(d, **kw), t)
    if params is not None:
        ds.set_parameters(*params)
    return ds


@gpu
def test_open_loop_costate_is_the_gradient_of_a_tracking_cost(lib):
    """pend_on_cart1 (no kinematic inputs): z[0] of l_dx[k] = X[k] - Xref[k], m_dx = X[K] - Xref[K] over the
    linearization of a simulated rollout equals d/dX[0] of J = sum_k |X[k] - Xref[k]|^2 / 2 (k = 0..K), the central
    difference taken through DSystem.simulate with all 2 nX perturbed rollouts in one batch."""
    d = G.desc("pend_on_cart1")
    K = 60
    ds = _dsys(d, np.arange(K + 1) * 0.01)
    nX = ds.nX
    rng = np.random.default_rng(5)
    X0 = np.array([0.1, 0.4, 0.0, 0.0])
    U = 0.5 * rng.normal(size=(1, K, ds.nU))
    X = ds.simulate(X0[None], U)[0]
    Xref = X + 0.1 * rng.normal(size=X.shape)
    J = lambda Xs: 0.5 * np.sum((Xs - Xref) ** 2, axis=(-2, -1))
    A, B = ds.linearize_trajectory(X, U[0])
    z = lib.adjoint_sweep(A, B, X[K] - Xref[K], X[:K] - Xref[:K])
    delta = 1e-5
    P = np.concatenate([X0 + delta * np.eye(nX), X0 - delta * np.eye(nX)])
    Js = J(ds.simulate(P, np.repeat(U, 2 * nX, axis=0)))
    grad = (Js[:nX] - Js[nX:]) / (2 * delta)
    assert np.max(np.abs(z[0] - grad)) <= 1e-6 * np.max(np.abs(grad)), (z[0], grad)


def _model(ds, X, U, seed):
    """A tracking cost's LQ model along (X, U): q [R,K+1,nX], r [R,K,nU], Q, S, R shared."""
    rng = np.random.default_rng(seed)
    Rn, K = X.shape[0], X.shape[1] - 1
    nX, nU = ds.nX, ds.nU
    q = X - (X + 0.05 * rng.normal(size=X.shape))
    r = 0.1 * U
    Q = np.broadcast_to(np.eye(nX), (K + 1, nX, nX)).copy()
    R = np.broadcast_to(0.1 * np.eye(nU), (K, nU, nU)).copy()
    return q, r, Q, None, R


def _composed(ds, X, U, q, r, Q, S, R, newton):
    """What calc_descent_direction replaces: calc_feedback_controller, calc_newton_model, lib.solve_tv_lq and the
    host loop (dproject with bdX = 0, bdU = -C)."""
    Kproj, A, B = ds.calc_feedback_controller(X, U, return_linearization=True)
    Rn, K = X.shape[0], X.shape[1] - 1
    z = None
    Qm, Sm, Rm = np.broadcast_to(Q, (Rn,) + Q.shape).copy(), np.zeros((Rn, K, ds.nX, ds.nU)), \
        np.broadcast_to(R, (Rn,) + R.shape).copy()
    if newton:
        z, xx, xu, uu = ds.calc_newton_model(X, U, A, B, Kproj, q[:, :K], r, q[:, K])
        Qm[:, :K] += xx
        Sm = Sm + xu
        Rm = Rm + uu
    Kl, C, _, _ = L.solve_tv_lq(A, B, q, r, Qm, Sm, Rm)
    dX, dU = ds.dproject(A, B, np.zeros(X.shape), -C, Kl)
    return Kproj, dX, dU, z


@gpu
@pytest.mark.parametrize("name,R,K", [("pend_on_cart1", 16, 100), ("puppet", 4, 20)], ids=["pend_on_cart1", "puppet"])
@pytest.mark.parametrize("newton", [False, True], ids=["steepest", "newton"])
def test_descent_direction_matches_the_composed_calls(lib, name, R, K, newton):
    d, g = G.desc(name), G.golden(name)
    t = np.arange(K + 1) * 0.01
    rng = np.random.default_rng(21)
    X, U = _traj(d, g, R, K, rng)
    ds = _dsys(d, t)
    q, r, Q, S, Rc = _model(ds, X, U, 3)
    out = ds.calc_descent_direction(X, U, q, r, Q, S, Rc, newton=newton, return_linearization=True)
    want = _composed(ds, X, U, q, r, Q, S, Rc, newton)
    assert len(out) == (6 if newton else 5)
    assert out[0].tobytes() == want[0].tobytes(), "Kproj"
    G.assert_close(out[1], want[1], name + " dX")
    G.assert_close(out[2], want[2], name + " dU")
    if newton:
        G.assert_close(out[3], want[3], name + " z")
    A, B = ds.linearize_trajectory(X, U)
    assert out[-2].tobytes() == A.tobytes() and out[-1].tobytes() == B.tobytes()
    # one trajectory without the rollout axis, and dx0
    dx0 = 1e-3 * rng.normal(size=ds.nX)
    one = ds.calc_descent_direction(X[1], U[1], q[1], r[1], Q, S, Rc, newton=newton, dx0=dx0)
    assert one[0].tobytes() == out[0][1].tobytes()
    assert one[1].shape == (K + 1, ds.nX) and one[2].shape == (K, ds.nU)
    assert np.array_equal(one[1][0], dx0)
    Kl, C, _, _ = L.solve_tv_lq(A[1], B[1], q[1], r[1], Q, np.zeros((K, ds.nX, ds.nU)), Rc) if not newton else (None,) * 4
    if not newton:
        # the loop that ends DOptimizer.calc_descent_direction, from dX[0] = dx0
        dX, dU = np.zeros((K + 1, ds.nX)), np.zeros((K, ds.nU))
        dX[0] = dx0
        for k in range(K):
            dU[k] = -(Kl[k] @ dX[k]) - C[k]
            dX[k + 1] = A[1, k] @ dX[k] + B[1, k] @ dU[k]
        G.assert_close(one[1], dX, name + " dX dx0")
        G.assert_close(one[2], dU, name + " dU dx0")


@gpu
def test_descent_direction_with_per_rollout_parameters(lib):
    """8 rollouts, each on its own parameter row: bitwise equal to one DSystem per rollout."""
    d, g = G.desc("pend_on_cart1"), G.golden("pend_on_cart1")
    R, K = 8, 30
    t = np.arange(K + 1) * 0.01
    rng = np.random.default_rng(17)
    refs = _refs(d)
    base = np.array([d.param_value(r) for r in refs])
    vals = base * rng.uniform(0.8, 1.2, (R, len(refs)))
    X, U = _traj(d, g, R, K, rng)
    ds = _dsys(d, t, (refs, vals))
    q, r, Q, S, Rc = _model(ds, X, U, 4)
    dx0 = 1e-3 * rng.normal(size=(R, ds.nX))
    got = ds.calc_descent_direction(X, U, q, r, Q, S, Rc, newton=True, dx0=dx0, return_linearization=True)
    for i in range(R):
        one = _dsys(d.with_params(refs, vals[i]), t)
        w = one.calc_descent_direction(X[i:i + 1], U[i:i + 1], q[i:i + 1], r[i:i + 1], Q, S, Rc, newton=True,
                                       dx0=dx0[i:i + 1], return_linearization=True)
        for k, (a, b) in enumerate(zip(got, w)):
            assert a[i:i + 1].tobytes() == b.tobytes(), "rollout %d output %d" % (i, k)
