"""The tracking cost on the device (trepb_track_batch*), the line-search candidates (trepb_candidates_batch*) and
discopt.DOptimizer, the batched optimiser built on them.

- The track kernel against numpy DCost loops: cost, dcost, q, r and the LQ model, with shared, per-rollout and
  indexed references, with and without the Newton blocks; q and r in the kernel's summation order bit for bit.
- A trajectory gives the same bits alone and inside batches of 37 and 1000.
- The candidates equal numpy's X + lam * dX bit for bit, with the gain copies.
- DOptimizer.step against the host composition it replaces (DSystem.calc_descent_direction with numpy model arrays,
  numpy cost and dcost, and the reference's one-candidate-at-a-time Armijo loop over DSystem.project).
- A rollout whose search fails gets a status and leaves the others alone; per-rollout parameters equal one
  DOptimizer per parameter row; optimize converges on a tracking problem with a feasible reference."""
import numpy as np
import pytest

import golden_util as G
from test_gpu_varied_deriv2 import _refs, _traj
from trep_b200 import discopt, lib as L, midpointvi as MV

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    if L.device_count() < 1:
        pytest.skip("needs a CUDA device")
    return L


def ordered_grad(d, W):
    """sum_i d[.., i] W[i, :] in ascending i with separately rounded products and sums: the kernel's order."""
    acc = np.zeros(d.shape[:-1] + (W.shape[1],))
    for i in range(W.shape[0]):
        acc = acc + d[..., i, None] * W[i]
    return acc


def numpy_track(X, U, Xd, Ud, Q, R, ref, dX=None, dU=None):
    """cost, dcost, q, r by DCost's methods and DOptimizer's loops, one trajectory at a time."""
    Bn, K = X.shape[0], X.shape[1] - 1
    cost, dcost = np.zeros(Bn), np.zeros(Bn)
    q, r = np.zeros(X.shape), np.zeros(U.shape)
    for b in range(Bn):
        c = discopt.DCost(Xd[ref[b]], Ud[ref[b]], Q, R)
        for k in range(K):
            cost[b] += c.l(X[b, k], U[b, k], k)
            q[b, k], r[b, k] = c.l_dx(X[b, k], U[b, k], k), c.l_du(X[b, k], U[b, k], k)
            if dX is not None:
                dcost[b] += q[b, k] @ dX[b, k] + r[b, k] @ dU[b, k]
        cost[b] += c.m(X[b, K])
        q[b, K] = c.m_dx(X[b, K])
        if dX is not None:
            dcost[b] += q[b, K] @ dX[b, K]
    return cost, dcost, q, r


def rel_close(a, b, what, rtol=1e-12):
    a, b = np.asarray(a), np.asarray(b)
    scale = max(float(np.max(np.abs(b))), 1e-300)
    assert np.all(np.abs(a - b) <= rtol * np.abs(b) + 1e-14 * scale), \
        "%s: max |a-b| = %.3e (max|b| = %.3e)" % (what, float(np.max(np.abs(a - b))), scale)


def spd(n, rng):
    A = rng.normal(size=(n, n))
    return A @ A.T / n + np.eye(n)


SHAPES = [(4, 1), (7, 3), (80, 18)]


@gpu
@pytest.mark.parametrize("nX,nU", SHAPES, ids=["4x1", "7x3", "80x18"])
@pytest.mark.parametrize("refs", ["shared", "per_rollout", "indexed"])
@pytest.mark.parametrize("newton", [False, True], ids=["quasi", "newton"])
def test_track_kernel_matches_numpy(lib, nX, nU, refs, newton):
    rng = np.random.default_rng(nX * 10 + nU)
    Bn, K = 5, 30
    X, U = rng.normal(size=(Bn, K + 1, nX)), rng.normal(size=(Bn, K, nU))
    nref = {"shared": 1, "per_rollout": Bn, "indexed": 3}[refs]
    Xd, Ud = rng.normal(size=(nref, K + 1, nX)), rng.normal(size=(nref, K, nU))
    ref = {"shared": np.zeros(Bn, int), "per_rollout": np.arange(Bn), "indexed": np.array([2, 0, 2, 1, 0])}[refs]
    Q, R = spd(nX, rng), spd(nU, rng)
    dX, dU = rng.normal(size=X.shape), rng.normal(size=U.shape)
    nt = (rng.normal(size=(Bn, K, nX, nX)), rng.normal(size=(Bn, K, nX, nU)), rng.normal(size=(Bn, K, nU, nU))) \
        if newton else None
    got = lib.track_cost(X, U, Xd if nref > 1 else Xd[0], Ud if nref > 1 else Ud[0], Q, R,
                         ref_index=None if refs == "shared" else ref, dX=dX, dU=dU, newton=nt)
    cost, dcost, q, r = numpy_track(X, U, Xd, Ud, Q, R, ref, dX, dU)
    rel_close(got["cost"], cost, "cost")
    rel_close(got["dcost"], dcost, "dcost")
    rel_close(got["q"], q, "q")
    rel_close(got["r"], r, "r")
    # in the kernel's summation order, bit for bit
    dx, du = X - Xd[ref], U - Ud[ref]
    assert got["q"].tobytes() == ordered_grad(dx, Q).tobytes()
    assert got["r"].tobytes() == ordered_grad(du, R).tobytes()
    assert got["l_dx"].tobytes() == got["q"][:, :K].tobytes() and got["m_dx"].tobytes() == got["q"][:, K].tobytes()
    # the model: DCost's second derivatives, plus the Newton blocks as the host sums them (Q[:, :K] += fdxdx)
    Qm = np.broadcast_to(Q, (Bn, K + 1, nX, nX)).copy()
    Sm, Rm = np.zeros((Bn, K, nX, nU)), np.broadcast_to(R, (Bn, K, nU, nU)).copy()
    if newton:
        Qm[:, :K] += nt[0]
        Sm = Sm + nt[1]
        Rm = Rm + nt[2]
    assert got["Qm"].tobytes() == Qm.tobytes()
    assert got["Sm"].tobytes() == Sm.tobytes()
    assert got["Rm"].tobytes() == Rm.tobytes()


@gpu
@pytest.mark.parametrize("nX,nU,big", [(7, 3, 1000), (80, 18, 37)], ids=["7x3", "80x18"])
def test_a_trajectory_gives_the_same_bits_alone_and_in_a_batch(lib, nX, nU, big):
    rng = np.random.default_rng(3)
    K = 25
    X, U = rng.normal(size=(big, K + 1, nX)), rng.normal(size=(big, K, nU))
    Xd, Ud = rng.normal(size=(4, K + 1, nX)), rng.normal(size=(4, K, nU))
    ref = rng.integers(0, 4, size=big)
    Q, R = spd(nX, rng), spd(nU, rng)
    dX, dU = rng.normal(size=X.shape), rng.normal(size=U.shape)
    nt = (rng.normal(size=(big, K, nX, nX)), rng.normal(size=(big, K, nX, nU)), rng.normal(size=(big, K, nU, nU)))
    run = lambda s: lib.track_cost(X[s], U[s], Xd, Ud, Q, R, ref_index=ref[s], dX=dX[s], dU=dU[s],
                                   newton=tuple(a[s] for a in nt))
    full = run(slice(0, big))
    for lo, hi in ((0, 1), (big - 1, big), (big // 2, big // 2 + 1), (1, 38) if big >= 38 else (0, big)):
        part = run(slice(lo, hi))
        for n in lib.TRACK_OUTPUTS:
            assert part[n].tobytes() == full[n][lo:hi].tobytes(), "%s rollouts %d:%d" % (n, lo, hi)


@gpu
def test_candidates_are_numpys_formula(lib):
    rng = np.random.default_rng(9)
    Rn, K, nX, nU, M = 6, 40, 7, 3, 8
    X, U, dX, dU = (rng.normal(size=s) for s in ((Rn, K + 1, nX), (Rn, K, nU), (Rn, K + 1, nX), (Rn, K, nU)))
    Kp = rng.normal(size=(Rn, K, nU, nX))
    lam = np.array([0.7 ** m for m in range(3, 3 + M)])
    for rows in (None, np.array([4, 1, 5], np.int32)):
        g = np.arange(Rn) if rows is None else rows
        bX, bU = np.zeros((g.size, M, K + 1, nX)), np.zeros((g.size, M, K, nU))
        Kc = np.zeros((g.size, M, K, nU, nX))
        lib.candidates_raw(False, 0, g.size, M, K, nX, nU, lam, X, U, dX, dU, Kp, bX, bU, Kc, rows=rows, nrollouts=Rn)
        for i, r in enumerate(g):
            for m in range(M):
                assert bX[i, m].tobytes() == (X[r] + lam[m] * dX[r]).tobytes()
                assert bU[i, m].tobytes() == (U[r] + lam[m] * dU[r]).tobytes()
                assert Kc[i, m].tobytes() == Kp[r].tobytes()


# ---- DOptimizer against the host composition ------------------------------------------------------------------
def _dsys(d, t, params=None):
    ds = discopt.DSystem(MV.MidpointVI(d), t)
    if params is not None:
        ds.set_parameters(*params)
    return ds


def _problem(name, R, K, seed):
    """Feasible rollouts (X, U) of `name` and a per-rollout reference near them."""
    d, g = G.desc(name), G.golden(name)
    t = np.arange(K + 1) * 0.01
    rng = np.random.default_rng(seed)
    X, U = _traj(d, g, R, K, rng)
    ds = _dsys(d, t)
    X = ds.simulate(X[:, 0], U)
    xd, ud = X + 0.02 * rng.normal(size=X.shape), U + 0.05 * rng.normal(size=U.shape)
    Q, Rw = np.diag(rng.uniform(0.5, 2.0, ds.nX)), np.diag(rng.uniform(0.05, 0.2, ds.nU))
    return d, t, ds, X, U, discopt.DCost(xd, ud, Q, Rw)


def host_model(ds, cost, X, U, method):
    """q, r in the kernel's order and Q, S, R as numpy arrays for DSystem.calc_descent_direction."""
    K = X.shape[1] - 1
    q, r = ordered_grad(X - cost.xd, cost.Q), ordered_grad(U - cost.ud, cost.R)
    if method == "steepest":
        Q, R = np.broadcast_to(np.eye(ds.nX), (K + 1, ds.nX, ds.nX)), np.broadcast_to(np.eye(ds.nU), (K, ds.nU, ds.nU))
    else:
        Q, R = np.broadcast_to(cost.Q, (K + 1, ds.nX, ds.nX)), np.broadcast_to(cost.R, (K, ds.nU, ds.nU))
    return q, r, np.ascontiguousarray(Q), None, np.ascontiguousarray(R)


def host_cost(cost, X, U):
    return numpy_track(X, U, cost.xd, cost.ud, cost.Q, cost.R, np.arange(X.shape[0]))[0]


def host_step(opt, X, U, method):
    """The reference's step on the host: direction, cost0 / dcost0 by numpy loops, one candidate at a time."""
    ds, cost = opt.dsys, opt.cost
    Kp, dX, dU = ds.calc_descent_direction(X, U, *host_model(ds, cost, X, U, method), newton=method == "newton")[:3]
    _, dcost0, _, _ = numpy_track(X, U, cost.xd, cost.ud, cost.Q, cost.R, np.arange(X.shape[0]), dX, dU)
    cost0 = host_cost(cost, X, U)
    Xn, Un, c, ms = X.copy(), U.copy(), cost0.copy(), np.full(X.shape[0], -1)
    for b in range(X.shape[0]):
        if abs(dcost0[b]) < opt.descent_tolerance:
            continue
        one = discopt.DCost(cost.xd[b], cost.ud[b], cost.Q, cost.R)
        for m in range(opt.armijo_max_iterations):
            lam = opt.armijo_beta ** m
            max_cost = cost0[b] + opt.armijo_alpha * lam * dcost0[b]
            try:
                nX, nU = ds.project(X[b] + lam * dX[b], U[b] + lam * dU[b], Kp[b], use_hint=False)
            except MV.ConvergenceError:
                continue
            cost1 = host_cost(discopt.DCost(one.xd[None], one.ud[None], one.Q, one.R), nX[None], nU[None])[0]
            if cost1 < max_cost:
                Xn[b], Un[b], c[b], ms[b] = nX, nU, cost1, m
                break
    return (Kp, dX, dU), dcost0, Xn, Un, c, ms


@gpu
@pytest.mark.parametrize("name,R,K", [("pend_on_cart1", 16, 100), ("puppet", 4, 20)], ids=["pend_on_cart1", "puppet"])
@pytest.mark.parametrize("method", ["steepest", "quasi", "newton"])
def test_step_matches_the_host_loop(lib, name, R, K, method):
    d, t, ds, X, U, cost = _problem(name, R, K, 11)
    opt = discopt.DOptimizer(ds, cost)
    direction = opt.calc_descent_direction(X, U, method)
    want_dir, dcost0, Xw, Uw, cw, mw = host_step(opt, X, U, method)
    for a, b, what in zip(direction, want_dir, ("Kproj", "dX", "dU")):
        assert a.tobytes() == b.tobytes(), what
    conv, Xn, Un, dc, c = opt.step(0, X, U, method)
    rel_close(dc, dcost0, "dcost0")
    assert np.array_equal(opt.last_armijo_m, mw), (opt.last_armijo_m, mw)
    assert np.any(mw >= 0), "some rollout should find a step on this problem"
    assert Xn.tobytes() == Xw.tobytes() and Un.tobytes() == Uw.tobytes()
    rel_close(c, cw, "cost")
    rel_close(opt.calc_cost(X, U), host_cost(cost, X, U), "calc_cost")
    rel_close(opt.calc_dcost(X, U, want_dir[1], want_dir[2]), dcost0, "calc_dcost")
    # one trajectory without the rollout axis
    one = discopt.DOptimizer(ds, discopt.DCost(cost.xd[2], cost.ud[2], cost.Q, cost.R))
    s1 = one.step(0, X[2], U[2], method)
    assert s1.X.tobytes() == Xn[2].tobytes() and s1.U.tobytes() == Un[2].tobytes() and s1.cost == c[2]


@gpu
def test_a_failed_search_leaves_the_other_rollouts_alone(lib):
    d, t, ds, X, U, cost = _problem("pend_on_cart1", 6, 60, 12)
    opt = discopt.DOptimizer(ds, cost)
    Kp, dX, dU = opt.calc_descent_direction(X, U, "quasi")
    good = opt.armijo_search(X, U, Kp, dX, dU)
    assert np.all(opt.last_status == discopt.STEP_ACCEPTED)
    m_good = opt.last_armijo_m.copy()
    bX, bU = dX.copy(), dU.copy()
    bX[0], bU[0] = -dX[0], -dU[0]       # rollout 0 now searches along an ascent direction
    bad = opt.armijo_search(X, U, Kp, bX, bU)
    assert opt.last_status[0] == discopt.ARMIJO_FAILED and opt.last_armijo_m[0] == -1
    assert np.all(opt.last_status[1:] == discopt.STEP_ACCEPTED)
    assert np.array_equal(opt.last_armijo_m[1:], m_good[1:])
    assert bad.nX[0].tobytes() == X[0].tobytes() and bad.nU[0].tobytes() == U[0].tobytes()
    assert bad.cost[0] == opt.calc_cost(X, U)[0]
    assert bad.nX[1:].tobytes() == good.nX[1:].tobytes() and bad.nU[1:].tobytes() == good.nU[1:].tobytes()
    assert bad.cost[1:].tobytes() == good.cost[1:].tobytes()
    # one trajectory without the rollout axis raises like the reference
    one = discopt.DOptimizer(ds, discopt.DCost(cost.xd[0], cost.ud[0], cost.Q, cost.R))
    with pytest.raises(MV.ConvergenceError, match="Armijo"):
        one.armijo_search(X[0], U[0], Kp[0], bX[0], bU[0])


@gpu
def test_per_rollout_parameters_equal_one_optimizer_per_row(lib):
    d, t, ds0, X, U, cost = _problem("pend_on_cart1", 8, 40, 13)
    rng = np.random.default_rng(14)
    refs = _refs(d)
    base = np.array([d.param_value(r) for r in refs])
    vals = base * rng.uniform(0.9, 1.1, (8, len(refs)))
    ds = _dsys(d, t, (refs, vals))
    X = ds.simulate(X[:, 0], U)          # each rollout feasible on its own parameter row
    opt = discopt.DOptimizer(ds, cost)
    for method in ("quasi", "newton"):
        got = opt.step(0, X, U, method)
        st, ms = opt.last_status.copy(), opt.last_armijo_m.copy()
        assert np.any(st == discopt.STEP_ACCEPTED), st
        for i in range(8):
            # one rollout with the rollout axis: a failed search is a status there, as in the batch
            one = discopt.DOptimizer(_dsys(d.with_params(refs, vals[i]), t),
                                     discopt.DCost(cost.xd[i:i + 1], cost.ud[i:i + 1], cost.Q, cost.R))
            w = one.step(0, X[i:i + 1], U[i:i + 1], method)
            assert got.X[i].tobytes() == w.X[0].tobytes() and got.U[i].tobytes() == w.U[0].tobytes(), (method, i)
            assert got.cost[i] == w.cost[0] and got.dcost[i] == w.dcost[0], (method, i)
            assert st[i] == one.last_status[0] and ms[i] == one.last_armijo_m[0], (method, i)


@gpu
def test_optimize_converges_on_a_feasible_reference(lib):
    d = G.desc("pend_on_cart1")
    R, K = 8, 100
    t = np.arange(K + 1) * 0.01
    ds = _dsys(d, t)
    rng = np.random.default_rng(15)
    X0 = np.tile([0.0, 0.3, 0.0, 0.0], (R, 1)) + 0.05 * rng.normal(size=(R, ds.nX))
    Ud = 0.5 * np.sin(np.linspace(0, 3, K))[None, :, None] * rng.uniform(0.5, 1.5, (R, 1, ds.nU))
    Xd = ds.simulate(X0, Ud)
    cost = discopt.DCost(Xd, Ud, np.eye(ds.nX), 0.1 * np.eye(ds.nU))
    U = Ud + 0.3 * rng.normal(size=Ud.shape)
    X = ds.simulate(X0, U)
    opt = discopt.DOptimizer(ds, cost)
    # the cost falls at every step of every rollout
    c = opt.calc_cost(X, U)
    Xs, Us = X, U
    for i in range(10):
        conv, Xs, Us, dc, cn = opt.step(i, Xs, Us, "quasi")
        st = opt.last_status
        assert not np.any(st == discopt.ARMIJO_FAILED), (i, st)
        moved = st == discopt.STEP_ACCEPTED
        assert i > 0 or np.all(moved)
        assert np.all(dc[moved] < 0) and np.all(cn[moved] < c[moved]), (i, cn, c)
        assert np.array_equal(cn[~moved], c[~moved])     # a converged rollout keeps its trajectory and cost
        c = cn
        if np.all(conv):
            break
    converged, Xo, Uo = opt.optimize(X, U, max_steps=50)
    assert np.all(converged), opt.last_status
    assert np.all(opt.last_status == discopt.STEP_CONVERGED)
    Kp, dX, dU = opt.calc_descent_direction(Xo, Uo, "newton")
    assert np.all(np.abs(opt.calc_dcost(Xo, Uo, dX, dU)) < opt.descent_tolerance)
    assert np.all(opt.calc_cost(Xo, Uo) < opt.calc_cost(X, U))
