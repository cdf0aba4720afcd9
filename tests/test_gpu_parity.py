"""GPU parity tests: the CUDA path, called through the C ABI (libtrepb.so), against
  (a) the committed golden vectors recorded from the reference itself, and
  (b) on seeded random batches, this library's results at commit f731ca3, which these tests then checked
      against the reference run live (tests/golden/expected/, see golden_util.expected).

Bar (BASELINE.json north_star): 1e-10 relative in fp64, identical Newton iteration counts.
Iteration counts can legitimately flip by one when an iterate lands within rounding distance of
the 1e-10 convergence threshold (SURVEY.md section 7, "iteration-count parity"); the tests
therefore require identical counts on the golden cases and bound the flip fraction on the
random batches, checking that flipped instances still agree to 1e-10.
"""
import os

import numpy as np
import pytest

import golden_util as G
from test_lq_reference import lq_pinned_cases, lqr_pinned_cases

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from trep_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


# LinearSpring / LinearDamper, PointOnPlane, wrenches: thread-per-instance kernels only
COOP_UNSUPPORTED = set()     # every plugin kind runs on the cooperative kernels since round 2


def _systems(lib, name):
    """(label, System) for every kernel flavour that can run the system: the specialised kernel
    (if one exists), the table-driven thread-per-instance kernel and the cooperative
    (warp-per-instance, shared-memory workspace) kernel."""
    d = G.desc(name)
    out = []
    s = lib.System(d)
    if s.specialized:
        out.append(("spec", s))
        # the instantiation with run-time parameters (for four systems lib.System picks the all-literal one)
        out.append(("spec-param", lib.System(d, literal=False)))
        assert out[-1][1].specialized
    out.append(("general", lib.System(d, specialize=False, cooperative=False)))
    if name not in COOP_UNSUPPORTED:
        c = lib.System(d, specialize=False, cooperative=True)
        assert c.cooperative and c.kernel_name == "cooperative"
        out.append(("coop", c))
        c = lib.System(d, cooperative=True)
        if c.kernel_name != "cooperative":      # a compile-time-size flavour exists for this shape
            if c.kernel_name.endswith("/ext"):      # external-slab layout: the default where it was built
                assert c.kernel_name == "cooperative/" + name + "/ext"
                out.append(("coop-static-ext", c))
                c = lib.System(d, cooperative=True, coop_two_warps=True)
                assert c.kernel_name == "cooperative/" + name + "/pair"
                out.append(("coop-static-pair", c))
                c = lib.System(d, cooperative=True, coop_one_warp=True)
            assert c.kernel_name == "cooperative/" + name
            out.append(("coop-static", c))
    return out


@pytest.mark.parametrize("name", G.ALL)
def test_golden_cases(lib, name):
    g = G.golden(name)
    for label, s in _systems(lib, name):
        if name in G.SMALL and name != "pendulum5":
            assert label != "spec" or s.specialized
        out = s.linearize(g["case_q1"], g["case_p1"], g["case_u1"], g["case_k2"], t1=g["case_t1"],
                          t2=g["case_t2"], q2_guess=g["case_q2_guess"],
                          lambda_guess=g["case_lambda_guess"], want_raw=True)
        assert np.all(out["status"] == 0), (label, out["status"])
        for k in ("q2", "p2", "lambda1", "A", "B"):
            G.assert_close(out[k], g["case_" + k], "%s[%s] %s" % (name, label, k))
        for k in G.RAW:
            G.assert_close(out[k], g["case_" + k], "%s[%s] %s" % (name, label, k))
        assert np.array_equal(out["iters"], g["case_iters"]), (label, out["iters"], g["case_iters"])


@pytest.mark.parametrize("name", G.SMALL)
def test_golden_rollout(lib, name):
    g = G.golden(name)
    if "roll_q" not in g:
        pytest.skip("no rollout recorded")
    dt, nsteps, sample = float(g["roll_dt"]), int(g["roll_nsteps"]), int(g["roll_sample"])
    for label, s in _systems(lib, name):
        p0 = s.calc_p2(dt, g["roll_q0"], g["roll_q1"])
        G.assert_close(p0[0], g["roll_p_init"], name + " p_init")
        u = None
        if s.nu:
            t = dt * (1 + np.arange(nsteps))
            u = np.stack([1.5 * np.sin(2.0 * t)] + [0.2 * np.cos(t)] * (s.nu - 1), axis=1)[None]
        out = s.step(g["roll_q1"], p0, dt, dt, nsteps=nsteps, u1=u, sample_every=sample)
        assert out["status"][0] == 0
        ns = nsteps // sample
        # early samples are tight; chaotic growth of rounding differences loosens later ones
        G.assert_close(out["traj_q"][0, 0], g["roll_q"][1], "%s[%s] first sample q" % (name, label), rtol=1e-9)
        G.assert_close(out["traj_q"][0, :ns], g["roll_q"][1:1 + ns], "%s[%s] traj q" % (name, label), rtol=1e-6)
        G.assert_close(out["traj_p"][0, :ns], g["roll_p"][1:1 + ns], "%s[%s] traj p" % (name, label), rtol=1e-6)
        assert abs(int(out["iters"][0]) - int(g["roll_iters"].sum())) <= max(2, nsteps // 100)


@pytest.mark.parametrize("coop", [True, False])
def test_puppet_rollout(lib, coop):
    g = G.golden("puppet")
    s = lib.System(G.desc("puppet"), cooperative=coop)
    assert s.cooperative == coop
    dt, nsteps = float(g["roll_dt"]), int(g["roll_nsteps"])
    p0 = s.calc_p2(dt, g["roll_q0"], g["roll_q1"])
    G.assert_close(p0[0], g["roll_p"][0], "puppet p_init")
    out = s.step(g["roll_q1"], p0, dt, dt, nsteps=nsteps, k2=g["roll_k2"][None], sample_every=1)
    assert out["status"][0] == 0
    G.assert_close(out["traj_q"][0], g["roll_q"][1:], "puppet traj q", rtol=1e-8)
    G.assert_close(out["traj_p"][0], g["roll_p"][1:], "puppet traj p", rtol=1e-8)
    G.assert_close(out["lambda1"][0], g["roll_lambda"][-1], "puppet lambda", rtol=1e-8)
    assert int(out["iters"][0]) == int(g["roll_iters"].sum())


RANDOM = {
    #  name            B    q-range  p-scale u-scale
    "damped_pendulum": (512, np.pi, 5.0, 0.0),
    "pendulum1": (256, np.pi, 2.0, 0.0),
    "pendulum5": (64, np.pi, 2.0, 0.0),
    "pend_on_cart1": (512, np.pi, 3.0, 2.0),
    "pend_on_cart2": (256, np.pi, 3.0, 2.0),
    "dual_pendulums": (512, np.pi, 3.0, 0.0),
}


@pytest.mark.parametrize("name", sorted(RANDOM))
def test_random_batch_vs_reference(lib, name):
    """Seeded random batch, ragged size (not a multiple of the warp or CTA size)."""
    B, qr, ps, us = RANDOM[name]
    B += 3
    rng = np.random.default_rng(1234)
    d = G.desc(name)
    nq, nd, nu = d.nq, d.nd, d.nu
    q1 = rng.uniform(-qr, qr, (B, nq))
    p1 = rng.normal(0, ps, (B, nd))
    u1 = rng.uniform(-us, us, (B, nu))
    k2 = np.zeros((B, 0))
    t1 = rng.uniform(0, 5, B)
    t2 = t1 + 0.01
    want = G.expected("random_batch_" + name, lambda: G.library_cases(name, t1, t2, q1, p1, u1, k2))
    for label, s in _systems(lib, name):
        out = s.linearize(q1, p1, u1, k2, t1=t1, t2=t2)
        assert np.array_equal(out["status"], want["status"])
        G.assert_cases_close(out, want, ("q2", "p2", "A", "B"), "%s[%s]" % (name, label))
        flips = int(np.sum(out["iters"] != want["iters"]))
        assert flips <= max(1, B // 100), "%s[%s]: %d/%d iteration counts differ" % (name, label, flips, B)


def test_puppet_random_vs_reference(lib):
    """Marionette: perturbed points of the golden trajectory (A and B compared on 4 of the 45 instances)."""
    g = G.golden("puppet")
    rng = np.random.default_rng(7)
    nd = G.desc("puppet").nd
    B = 45          # ragged: not a multiple of the 8 instances a CTA of the cooperative kernel takes per round
    idx = rng.integers(1, 58, B)
    q1 = g["roll_q"][idx].copy()
    p1 = g["roll_p"][idx].copy()
    q1[:, :nd] += rng.normal(0, 0.02, (B, nd))
    p1 += rng.normal(0, 0.02, (B, nd))
    k2 = g["roll_k2"][idx]          # kinematic configs at the end of step idx -> idx+1
    lam = g["roll_lambda"][idx - 1]
    t1 = 0.01 * (idx + 1)
    t2 = t1 + 0.01
    want = G.expected("puppet_random", lambda: G.library_cases("puppet", t1, t2, q1, p1, np.zeros((B, 0)), k2,
                                                               lambda_guess=lam, m=4))
    for coop in (True, False):
        s = lib.System(G.desc("puppet"), cooperative=coop)
        assert s.cooperative == coop
        out = s.linearize(q1, p1, None, k2, t1=t1, t2=t2, lambda_guess=lam)
        assert np.array_equal(out["status"], want["status"])
        ok = want["status"] == 0
        G.assert_cases_close(out, want, ("q2", "p2", "lambda1", "A", "B"), "puppet[coop=%s]" % coop)
        assert np.array_equal(out["iters"][ok], want["iters"][ok])


def test_device_pointer_entry_points_match_host(lib):
    """*_dev entry points (inputs resident in HBM) give the same bits as the host entry points."""
    g = G.golden("pend_on_cart1")
    s = lib.System(G.desc("pend_on_cart1"))
    B = 1000
    rng = np.random.default_rng(3)
    q1 = rng.uniform(-3, 3, (B, 2)); p1 = rng.normal(0, 3, (B, 2)); u1 = rng.uniform(-2, 2, (B, 1))
    host = s.linearize(q1, p1, u1, None, t1=0.0, dt=0.01)
    db = lambda a: lib.DeviceBuffer(0, a.shape, a.dtype).upload(a)
    dq, dp, du = db(q1), db(p1), db(u1)
    dA = lib.DeviceBuffer(0, (B, 4, 4)); dB = lib.DeviceBuffer(0, (B, 4, 1))
    dq2 = lib.DeviceBuffer(0, (B, 2)); dp2 = lib.DeviceBuffer(0, (B, 2))
    dit = lib.DeviceBuffer(0, (B,), np.int32); dst = lib.DeviceBuffer(0, (B,), np.int32)
    s.linearize_raw(True, B, dq, dp, du, None, dst, t1_scalar=0.0, dt_scalar=0.01, q2=dq2, p2=dp2,
                    iters=dit, A=dA, B=dB)
    lib.synchronize(0)
    assert s.last_kernel_ms() > 0
    assert np.array_equal(dA.download(), host["A"])
    assert np.array_equal(dB.download(), host["B"])
    assert np.array_equal(dq2.download(), host["q2"])
    assert np.array_equal(dit.download(), host["iters"])
    assert np.all(dst.download() == 0)


def test_status_codes_not_converged_and_empty_batch(lib):
    s = lib.System(G.desc("damped_pendulum"))
    # max_iterations = 0 with a start far from the root: the reference raises ConvergenceError
    # after exceeding max_iterations (midpointvi.c:715-718); here: status -1, batch continues
    q1 = np.array([[0.5], [0.0]]); p1 = np.array([[40.0], [0.0]])
    out = s.step(q1, p1, 0.0, 0.01, max_iterations=0)
    assert out["status"][0] == -1
    # second instance: q=0,p=0 is an exact fixed point -> converged with 0 iterations
    assert out["status"][1] == 0 and out["iters"][1] == 0
    out = s.step(np.zeros((0, 1)), np.zeros((0, 1)), 0.0, 0.01)
    assert out["q2"].shape == (0, 1)


def test_full_size_properties(lib):
    """BASELINE config 2 at full width (2^20 damped pendulums), size-independent properties:
    duplicated instances give identical bits wherever they sit in the batch, and a long rollout
    equals the same rollout split into two launches (restartability)."""
    s = lib.System(G.desc("damped_pendulum"))
    B = 1 << 20
    rng = np.random.default_rng(0)
    th0 = rng.uniform(-np.pi, np.pi, 1024)
    th1 = th0 + rng.uniform(-0.02, 0.02, 1024)
    q0 = np.tile(th0, B // 1024)[:, None]
    q1 = np.tile(th1, B // 1024)[:, None]
    p = s.calc_p2(0.01, q0, q1)
    a = s.step(q1, p, 0.01, 0.01, nsteps=40)
    assert np.all(a["status"] == 0)
    qq = a["q2"].reshape(B // 1024, 1024)
    assert np.all(qq == qq[0]), "same inputs must give the same bits at every batch position"
    b1 = s.step(q1[:4096], p[:4096], 0.01, 0.01, nsteps=15)
    b2 = s.step(b1["q2"], b1["p2"], 0.01 + 15 * 0.01, 0.01, nsteps=25)
    # t0 differs by rounding between one 40-step launch and 15+25 -> compare to 1e-12
    G.assert_close(b2["q2"], a["q2"][:4096], "split rollout q", rtol=1e-12)
    G.assert_close(b2["p2"], a["p2"][:4096], "split rollout p", rtol=1e-12)
    assert np.array_equal(b1["iters"] + b2["iters"], a["iters"][:4096]) or \
        np.mean(b1["iters"] + b2["iters"] != a["iters"][:4096]) < 1e-3


D2_SYSTEMS = ["tase_pendulum", "pendulum1", "pendulum5", "damped_pendulum", "pend_on_cart1", "pend_on_cart2"]


@pytest.mark.parametrize("name", D2_SYSTEMS)
def test_golden_second_derivatives(lib, name):
    """Every second-derivative tensor against the reference's _calc_deriv2 (golden cases)."""
    g = G.golden(name)
    flavours = _systems(lib, name) + [("general/pairwise", lib.System(G.desc(name), specialize=False, cooperative=False,
                                                                     d2_pairwise=True))]
    for label, s in flavours:
        out = s.deriv2(g["case_q1"], g["case_p1"], g["case_u1"], g["case_k2"], t1=g["case_t1"],
                       t2=g["case_t2"], q2_guess=g["case_q2_guess"], lambda_guess=g["case_lambda_guess"])
        assert np.all(out["status"] == 0)
        G.assert_close(out["A"], g["case_A"], "%s[%s] A" % (name, label))
        G.assert_d2_close(out, g, "%s[%s]" % (name, label))


def test_puppet_second_derivatives(lib):
    """Marionette (nd 22, nk 18, nc 6): all 30 tensors of one golden case (1.76 MB of doubles)."""
    g = G.golden("puppet")
    g2 = G.puppet_deriv2()
    c = int(g2["case_index"][0])
    sl = slice(c, c + 1)
    # the second-derivative kernel consumes the factorizations the linearize kernel exports:
    # check both producers (cooperative and thread-per-instance) and both second-derivative schemes
    # (dual Jacobian tables per parameter + contraction; hyper-dual residual per parameter pair)
    for coop, pairwise in ((True, False), (False, False), (True, True)):
        s = lib.System(G.desc("puppet"), cooperative=coop, d2_pairwise=pairwise)
        out = s.deriv2(g["case_q1"][sl], g["case_p1"][sl], None, g["case_k2"][sl], t1=g["case_t1"][sl],
                       t2=g["case_t2"][sl], q2_guess=g["case_q2_guess"][sl], lambda_guess=g["case_lambda_guess"][sl])
        assert out["status"][0] == 0
        G.assert_d2_close(out, g2, "puppet[coop=%s pairwise=%s]" % (coop, pairwise))


def test_puppet_second_derivative_schemes_agree_on_a_ragged_batch(lib):
    """Marionette, ragged batch with one instance that cannot converge (status != 0 must be skipped,
    not abort the batch): the per-parameter scheme (dual Jacobian tables + contraction) and the
    per-pair scheme (hyper-dual residual) give the same tensors and the same z-contracted forms."""
    g = G.golden("puppet")
    d = G.desc("puppet")
    rng = np.random.default_rng(5)
    B = 37
    idx = rng.integers(1, g["roll_q"].shape[0] - 1, B)
    q1 = g["roll_q"][idx].copy(); p1 = g["roll_p"][idx].copy()
    q1[:, :d.nd] += rng.normal(0, 0.01, (B, d.nd)); p1 += rng.normal(0, 0.01, (B, d.nd))
    k2 = g["roll_k2"][idx].copy(); lam = g["roll_lambda"][idx - 1].copy()
    q1[3] = np.nan      # a broken instance
    z = rng.normal(0, 1, (B, d.nX))
    outs = []
    for pairwise in (False, True):
        s = lib.System(d, d2_pairwise=pairwise)
        outs.append(s.deriv2(q1, p1, None, k2, t1=0.0, dt=0.01, lambda_guess=lam, z=z))
    a, b = outs
    assert np.array_equal(a["status"], b["status"]) and a["status"][3] != 0
    ok = a["status"] == 0
    assert ok.sum() == B - 1
    for n in list(lib.System(d).d2_shapes(1)) + ["fdxdx", "fdxdu", "fdudu"]:
        x, y = a[n][ok], b[n][ok]
        if x.size == 0:
            continue
        assert np.max(np.abs(x - y)) <= 1e-9 * max(1.0, np.max(np.abs(y))), n
    # the z-contracted forms are the contraction of the tensors (dsystem.py:320-386)
    nq, nd = d.nq, d.nd
    i = int(np.flatnonzero(ok)[0])
    zz = z[i]
    want = np.einsum("abj,j->ab", a["q2_dq1dq1"][i], zz[:nd]) + np.einsum("abj,j->ab", a["p2_dq1dq1"][i], zz[nq:nq + nd])
    got = a["fdxdx"][i][:nq, :nq]
    assert np.max(np.abs(got - want)) <= 1e-10 * max(1.0, np.max(np.abs(want)))


def test_puppet_second_derivatives_across_batch_chunks(lib):
    """The per-parameter scheme processes a large batch in chunks (its table records are bounded to a
    few GB): replicas of the same instances spread over more than one chunk give identical results."""
    g = G.golden("puppet")
    d = G.desc("puppet")
    rng = np.random.default_rng(9)
    base = 5
    idx = rng.integers(1, g["roll_q"].shape[0] - 1, base)
    reps = 400                                   # 2000 instances: more than one 4 GB chunk of records
    til = lambda a: np.tile(a, (reps,) + (1,) * (a.ndim - 1))
    q1, p1, k2, lam = til(g["roll_q"][idx]), til(g["roll_p"][idx]), til(g["roll_k2"][idx]), til(g["roll_lambda"][idx - 1])
    z = til(rng.normal(0, 1, (base, d.nX)))
    s = lib.System(d)
    out = s.deriv2(q1, p1, None, k2, t1=0.0, dt=0.01, lambda_guess=lam, z=z, tensors=False)
    assert np.all(out["status"] == 0)
    for n in ("fdxdx", "fdxdu", "fdudu"):
        a = out[n].reshape((reps, base) + out[n].shape[1:])
        assert np.array_equal(a, np.broadcast_to(a[:1], a.shape)), n
    small = s.deriv2(q1[:base], p1[:base], None, k2[:base], t1=0.0, dt=0.01, lambda_guess=lam[:base], z=z[:base], tensors=False)
    assert np.array_equal(small["fdxdx"], out["fdxdx"][:base])


def test_second_derivatives_by_finite_differences_where_the_reference_has_none(lib):
    """dual_pendulums: the reference cannot run _calc_deriv2 here (LinearSpring has no C V_dqdqdq,
    potentials/linearspring.c); the tensors are checked against central differences of this
    library's own first derivatives instead."""
    s = lib.System(G.desc("dual_pendulums"))
    rng = np.random.default_rng(11)
    q1 = rng.uniform(-1, 1, (1, 2)); p1 = rng.normal(0, 1, (1, 2))
    out = s.deriv2(q1, p1, t1=0.0, dt=0.01)
    eps = 1e-6
    for a in range(2):
        dq = np.zeros((1, 2)); dq[0, a] = eps
        lp = s.linearize(q1 + dq, p1, t1=0.0, dt=0.01, want_raw=True, tolerance=1e-13)
        lm = s.linearize(q1 - dq, p1, t1=0.0, dt=0.01, want_raw=True, tolerance=1e-13)
        fd = (lp["q2_dq1"] - lm["q2_dq1"]) / (2 * eps)      # [1][b][out] = d/dq1_a of q2_dq1[b][out]
        assert np.max(np.abs(fd[0] - out["q2_dq1dq1"][0, a])) < 2e-6 * max(1.0, np.max(np.abs(fd)))
        fd = (lp["p2_dp1"] - lm["p2_dp1"]) / (2 * eps)
        assert np.max(np.abs(fd[0] - out["p2_dq1dp1"][0, a])) < 2e-6 * max(1.0, np.max(np.abs(fd)))


def test_singular_jacobian_status(lib):
    """A massless dynamic joint makes the DEL Jacobian singular: the reference raises ValueError from
    LU_decomp (math-code.c:393-398) -> ConvergenceError (midpointvi.py:198-201); here status -2."""
    from trep_b200 import model as M
    s = M.System()
    s.import_frames([M.rx("a"), [M.tz(-1.0)]])
    M.Gravity(s)
    h = lib.System(s.describe())
    out = h.step(np.array([[0.1], [0.2]]), np.array([[1.0], [0.0]]), 0.0, 0.01)
    assert out["status"][0] == -2
    assert out["status"][1] == 0 and out["iters"][1] == 0    # p = 0, no mass: already a solution


def _trajectory(lib, name, X0, U0, dt):
    """A feasible trajectory from X0 = [q; p] under the inputs U0 (what the reference's DSystem.set / step / f give)."""
    r = lib.System(G.desc(name)).step(X0[None, :2], X0[None, 2:], 0.0, dt, nsteps=len(U0), u1=U0[None], sample_every=1)
    return np.concatenate([X0[None], np.concatenate([r["traj_q"][0], r["traj_p"][0]], axis=1)])


@pytest.mark.parametrize("name", ["pend_on_cart1", "pend_on_cart2"])
def test_project_matches_reference(lib, name):
    """Closed-loop rollouts (trepb_project_batch) against the reference's DSystem.project: a batch of
    perturbed candidates around one trajectory, one shared gain sequence, every kernel flavour."""
    rng = np.random.default_rng(5)
    dt, K, R = 0.01, 40, 5
    t = dt * np.arange(K + 1)
    nX, nU = G.desc(name).nX, G.desc(name).nU
    # a feasible trajectory to perturb
    X0 = np.zeros(nX); X0[1] = 0.3
    U0 = 0.5 * np.sin(3 * t[:K])[:, None] * np.ones((1, nU))
    Kfb = rng.normal(0, 0.5, (K, nU, nX))
    dX, dU = rng.normal(0, 1e-2, (R, K + 1, nX)), rng.normal(0, 1e-2, (R, K, nU))

    def record():
        X = _trajectory(lib, name, X0, U0, dt)
        p = lib.System(G.desc(name)).project(X[None] + dX, U0[None] + dU, Kfb, 0.0, dt)
        return {"X": X, "pX": p["X"], "pU": p["U"]}
    want = G.expected("project_" + name, record)
    bX, bU = want["X"][None] + dX, U0[None] + dU
    for label, s in _systems(lib, name):
        out = s.project(bX, bU, Kfb, 0.0, dt)
        assert np.all(out["status"] == 0) and np.all(out["fail_step"] == K), label
        for r in range(R):
            G.assert_close(out["X"][r], want["pX"][r], "%s[%s] X of candidate %d" % (name, label, r), rtol=1e-9)
            G.assert_close(out["U"][r], want["pU"][r], "%s[%s] U of candidate %d" % (name, label, r), rtol=1e-9)
    # the DSystem mirror: same call as the reference's, batch or single candidate
    from trep_b200 import midpointvi as MV, discopt as DO
    d = DO.DSystem(MV.MidpointVI(G.desc(name)), t)
    got = d.project(bX[0], bU[0], Kfb)
    G.assert_close(got.X, want["pX"][0], name + " DSystem.project X", rtol=1e-9)
    G.assert_close(got.U, want["pU"][0], name + " DSystem.project U", rtol=1e-9)
    # armijo_simulate's variant (no hint) gives the same trajectory (to the Newton tolerance)
    nohint = lib.System(G.desc(name)).project(bX, bU, Kfb, 0.0, dt, use_hint=False)
    G.assert_close(nohint["X"], want["pX"], name + " no-hint X", rtol=1e-7)


def test_project_puppet_kinematic_feedback(lib):
    """Marionette: the inputs are the kinematic string configs (rho), so the feedback moves the
    strings.  Both table-driven flavours against the reference, and a failing candidate reports
    its first failed step instead of aborting the batch."""
    g = G.golden("puppet")
    rng = np.random.default_rng(9)
    dt, K = float(g["roll_dt"]), 10
    t = dt * (1 + np.arange(K + 1))
    d = G.desc("puppet")
    nX, nU, nq, nd = d.nX, d.nU, d.nq, d.nd
    # golden rollout as the nominal trajectory: X = [Q; p; v]
    Q, P = g["roll_q"], g["roll_p"]
    X = np.zeros((K + 1, nX))
    X[:, :nq] = Q[:K + 1]; X[:, nq:nq + nd] = P[:K + 1]
    X[1:, nq + nd:] = (Q[1:K + 1, nd:] - Q[:K, nd:]) / dt
    U = g["roll_k2"][:K].copy()              # rho[k] = kinematic configs at k+1
    # gains on the dynamic-configuration error only, and small: a string moved by eps in one step
    # changes the momenta by ~ m eps / dt, random gains on p or v make the closed loop blow up
    Kfb = np.zeros((K, nU, nX)); Kfb[:, :, :nd] = rng.normal(0, 2e-3, (K, nU, nd))
    R = 3
    bX = np.repeat(X[None], R, axis=0)
    tt = dt * np.arange(K)[None, :, None]
    bU = U[None] + 2e-4 * np.sin(40 * tt + rng.uniform(0, 6, (R, 1, nU)))   # candidates: wiggled strings
    want = G.expected("project_puppet", lambda: lib.System(d).project(bX, bU, Kfb, t[0], dt))
    for coop in (True, False):
        s = lib.System(G.desc("puppet"), cooperative=coop)
        out = s.project(bX, bU, Kfb, t[0], dt)
        assert np.all(out["status"] == 0)
        for r in range(R):
            G.assert_close(out["X"][r], want["X"][r], "puppet[coop=%s] X %d" % (coop, r), rtol=1e-7)
            G.assert_close(out["U"][r], want["U"][r], "puppet[coop=%s] U %d" % (coop, r), rtol=1e-7)
            assert np.max(np.abs(out["U"][r] - bU[r])) > 1e-6      # the feedback did something
    # a candidate that cannot be solved (strings pulled far away at step 5) fails alone
    bad = bU.copy()
    bad[1, 5] += 50.0
    out = lib.System(G.desc("puppet")).project(bX, bad, Kfb, t[0], dt, max_iterations=30)
    assert out["status"][1] != 0 and out["fail_step"][1] == 5
    assert out["status"][0] == 0 and out["status"][2] == 0
    G.assert_close(out["X"][0], want["X"][0], "puppet X next to a failing candidate", rtol=1e-7)


def test_lqr_sweep_matches_reference(lib):
    """trepb_lqr_batch against its own results pinned at f731ca3 (golden_util.expected), which were checked against
    the reference's discopt.dlqr.solve_tv_lqr (dlqr.py:9-38) run live: random stabilisable problems of the
    marionette's size and of pend-on-cart's, constant and per-step weights, several rollouts in one launch.  The inputs
    come from test_lq_reference, which holds the long-double reference of tests/lqref.py to the same pins."""
    for key, A, B, Qs, Rs in lqr_pinned_cases():
        nX = A.shape[2]
        Kg, Pg = lib.solve_tv_lqr(A, B, Qs, Rs)
        want = G.expected(key, lambda: {"K": Kg, "P": Pg})
        for r in range(A.shape[0]):
            G.assert_close(Kg[r], want["K"][r], "lqr gains nX=%d rollout %d" % (nX, r), rtol=1e-9)
            G.assert_close(Pg[r], want["P"][r], "lqr P0 nX=%d rollout %d" % (nX, r), rtol=1e-9)


def test_lq_sweep_matches_reference(lib):
    """trepb_lq_batch against its own results pinned at f731ca3 (golden_util.expected), which were checked against
    the reference's discopt.dlqr.solve_tv_lq (dlqr.py:41-81) run live: linear and cross cost terms, costs shared by the
    batch and one set per rollout, with and without S.  The inputs come from test_lq_reference, which holds the
    long-double reference of tests/lqref.py to the same pins."""
    for key, A, B, q, r, Qs, Ss, Rs, _ in lq_pinned_cases():
        nX = A.shape[2]
        Kg, Cg, Pg, bg = lib.solve_tv_lq(A, B, q, r, Qs, Ss, Rs)
        want = G.expected(key, lambda: {"K": Kg, "C": Cg, "P": Pg, "b": bg})
        for i in range(A.shape[0]):
            G.assert_close(Kg[i], want["K"][i], "lq gains nX=%d rollout %d" % (nX, i), rtol=1e-9)
            G.assert_close(Cg[i], want["C"][i], "lq affine term nX=%d rollout %d" % (nX, i), rtol=1e-9)
            G.assert_close(Pg[i], want["P"][i], "lq P0 nX=%d rollout %d" % (nX, i), rtol=1e-9)
            G.assert_close(bg[i], want["b"][i], "lq b0 nX=%d rollout %d" % (nX, i), rtol=1e-9)


def test_feedback_controller_pipeline(lib):
    """DSystem.calc_feedback_controller + project (dsystem.py:426-457, 474-494) end to end on the GPU
    (linearize_trajectory -> Riccati sweep -> closed-loop rollout) against the reference doing the
    same on the host, pend-on-cart."""
    from trep_b200 import midpointvi as MV, discopt as DO
    name = "pend_on_cart1"
    dt, K = 0.01, 50
    t = dt * np.arange(K + 1)
    X0 = np.zeros(G.desc(name).nX); X0[1] = 0.2
    U0 = 0.3 * np.sin(2 * t[:K])[:, None]
    noise = np.random.default_rng(2).normal(0, 1e-2, (K + 1, len(X0)))
    d = DO.DSystem(MV.MidpointVI(G.desc(name)), t)

    def record():
        X = _trajectory(lib, name, X0, U0, dt)
        Kfb = d.calc_feedback_controller(X, U0)
        p = d.project(X + noise, U0, Kfb)
        return {"X": X, "K": Kfb, "pX": p.X, "pU": p.U}
    want = G.expected("feedback_pipeline", record)
    X = want["X"]
    Kgpu = d.calc_feedback_controller(X, U0)
    G.assert_close(Kgpu, want["K"], "feedback gains", rtol=1e-8)
    got = d.project(X + noise, U0, Kgpu)
    G.assert_close(got.X, want["pX"], "projected X", rtol=1e-8)
    G.assert_close(got.U, want["pU"], "projected U", rtol=1e-8)


# ---- plugin kinds beyond BASELINE.json's configs (SURVEY 8f rank 4): PointOnPlane, wrenches ----------
@pytest.mark.parametrize("name", G.EXTRA)
def test_extra_plugin_kinds_golden_cases(lib, name):
    """PointOnPlane constraints (pccd) and Body / Hybrid / Spatial wrenches (wrench_arm): step, every
    first-derivative array, A / B and the Newton iteration counts against the reference."""
    g = G.golden(name)
    # the table-driven kernels, and the register-resident specialised ones where the build made them
    flavours = [("general", lib.System(G.desc(name), specialize=False, cooperative=False))]
    s = lib.System(G.desc(name))              # the library's own choice: a specialised thread kernel
    flavours.append(("default:" + s.kernel_name, s))   # (wrench_arm, spline_pendulum) or cooperative/pccd
    assert s.kernel_name == {"pccd": "cooperative/pccd"}.get(name, name)
    if name not in COOP_UNSUPPORTED:          # PointOnPlane is implemented by the cooperative kernels too
        flavours.append(("coop", lib.System(G.desc(name), specialize=False, cooperative=True)))
    for label, s in flavours:
        out = s.linearize(g["case_q1"], g["case_p1"], g["case_u1"], g["case_k2"], t1=g["case_t1"],
                          t2=g["case_t2"], q2_guess=g["case_q2_guess"],
                          lambda_guess=g["case_lambda_guess"], want_raw=True)
        assert np.all(out["status"] == 0)
        for k in ("q2", "p2", "lambda1", "A", "B"):
            G.assert_close(out[k], g["case_" + k], "%s[%s] %s" % (name, label, k))
        for k in G.RAW:
            G.assert_close(out[k], g["case_" + k], "%s[%s] %s" % (name, label, k))
        assert np.array_equal(out["iters"], g["case_iters"]), label


@pytest.mark.parametrize("pairwise", [False, True])
@pytest.mark.parametrize("name", G.EXTRA_D2)
def test_extra_plugin_kinds_second_derivatives(lib, name, pairwise):
    g = G.golden(name)
    for spec in (False, True, "coop"):
        if spec == "coop":
            if name in COOP_UNSUPPORTED:
                continue                  # the cooperative linearize kernel as producer of the factors
            s = lib.System(G.desc(name), d2_pairwise=pairwise, specialize=False, cooperative=True)
        else:
            s = lib.System(G.desc(name), d2_pairwise=pairwise, specialize=spec, cooperative=False)
        if spec is True and (not s.specialized or not pairwise):
            continue                      # a specialised system always uses the per-pair scheme
        out = s.deriv2(g["case_q1"], g["case_p1"], g["case_u1"], g["case_k2"], t1=g["case_t1"],
                       t2=g["case_t2"], q2_guess=g["case_q2_guess"], lambda_guess=g["case_lambda_guess"])
        assert np.all(out["status"] == 0)
        G.assert_d2_close(out, g, "%s[pairwise=%s spec=%s]" % (name, pairwise, spec))


def test_pccd_rollout(lib):
    """examples/pccd.py: 300 steps of the closed chain, every step against the reference."""
    g = G.golden("pccd")
    s = lib.System(G.desc("pccd"))
    dt, nsteps = float(g["roll_dt"]), int(g["roll_nsteps"])
    p0 = s.calc_p2(dt, g["roll_q0"], g["roll_q1"])
    G.assert_close(p0[0], g["roll_p"][0], "pccd p_init")
    out = s.step(g["roll_q1"], p0, dt, dt, nsteps=nsteps, sample_every=1)
    assert out["status"][0] == 0
    G.assert_close(out["traj_q"][0], g["roll_q"][1:], "pccd traj q", rtol=1e-7)
    G.assert_close(out["traj_p"][0], g["roll_p"][1:], "pccd traj p", rtol=1e-7)
    assert abs(int(out["iters"][0]) - int(g["roll_iters"].sum())) <= 3


def test_wrench_arm_rollout(lib):
    g = G.golden("wrench_arm")
    s = lib.System(G.desc("wrench_arm"))
    dt, nsteps, sample = float(g["roll_dt"]), int(g["roll_nsteps"]), int(g["roll_sample"])
    p0 = s.calc_p2(dt, g["roll_q0"], g["roll_q1"])
    G.assert_close(p0[0], g["roll_p_init"], "wrench_arm p_init")
    t = dt * (1 + np.arange(nsteps))
    u = np.stack([np.sin(3 * t), 0.5 * np.cos(2 * t), 0.8 * np.sin(t), 0.3 * np.cos(t), -0.6 * np.sin(2 * t)], axis=1)[None]
    out = s.step(g["roll_q1"], p0, dt, dt, nsteps=nsteps, u1=u, sample_every=sample)
    assert out["status"][0] == 0
    ns = nsteps // sample
    G.assert_close(out["traj_q"][0, :ns], g["roll_q"][1:1 + ns], "wrench_arm traj q", rtol=1e-7)
    G.assert_close(out["traj_p"][0, :ns], g["roll_p"][1:1 + ns], "wrench_arm traj p", rtol=1e-7)
    assert abs(int(out["iters"][0]) - int(g["roll_iters"].sum())) <= 4


@pytest.mark.parametrize("name", G.EXTRA)
def test_extra_plugin_kinds_random_vs_reference(lib, name):
    """Seeded ragged batches (pinned results, golden_util.expected)."""
    rng = np.random.default_rng(21)
    d = G.desc(name)
    nq, nd, nu = d.nq, d.nd, d.nu
    B = 67
    if name == "pccd":
        g = G.golden("pccd")
        idx = rng.integers(1, g["roll_q"].shape[0] - 1, B)
        q1 = g["roll_q"][idx] + rng.normal(0, 0.01, (B, nq))
        p1 = g["roll_p"][idx] + rng.normal(0, 0.05, (B, nd))
        lam = g["roll_lambda"][idx - 1]
    elif name == "spline_pendulum":
        q1 = np.stack([rng.uniform(-2.4, 2.2, B), rng.uniform(-np.pi, np.pi, B)], axis=1)
        p1 = rng.normal(0, 1.0, (B, nd))
        lam = None
    else:
        q1 = np.stack([rng.uniform(-np.pi, np.pi, B), rng.uniform(-1.2, 1.2, B), rng.uniform(-0.3, 0.5, B)], axis=1)
        p1 = rng.normal(0, 1.0, (B, nd))
        lam = None
    u1 = rng.uniform(-2, 2, (B, nu))
    k2 = np.zeros((B, 0))
    t1 = rng.uniform(0, 5, B)
    t2 = t1 + 0.01
    want = G.expected("extra_random_" + name, lambda: G.library_cases(name, t1, t2, q1, p1, u1, k2, lambda_guess=lam))
    s = lib.System(G.desc(name))
    out = s.linearize(q1, p1, u1, k2, t1=t1, t2=t2, lambda_guess=lam)
    assert np.array_equal(out["status"], want["status"])
    G.assert_cases_close(out, want, ("q2", "p2", "lambda1", "A", "B"), name)
    assert int(np.sum(out["iters"] != want["iters"])) <= 1


@pytest.mark.parametrize("pairwise", [False, True])
def test_spline_spring_second_derivatives_by_finite_differences(lib, pairwise):
    """NonlinearConfigSpring: the reference's V_dqdqdq has a sign error
    (potentials/nonlinear_config_spring.c:53), so its second-derivative tensors cannot serve as the
    oracle for this plugin; both schemes are checked against central differences of this library's own
    first derivatives (which match the reference) instead."""
    s = lib.System(G.desc("spline_pendulum"), d2_pairwise=pairwise, specialize=False)
    rng = np.random.default_rng(3)
    q1 = np.array([[0.45, -0.3]]); p1 = rng.normal(0, 1, (1, 2))
    out = s.deriv2(q1, p1, t1=0.0, dt=0.01)
    eps = 1e-6
    for a in range(2):
        dq = np.zeros((1, 2)); dq[0, a] = eps
        lp = s.linearize(q1 + dq, p1, t1=0.0, dt=0.01, want_raw=True, tolerance=1e-13)
        lm = s.linearize(q1 - dq, p1, t1=0.0, dt=0.01, want_raw=True, tolerance=1e-13)
        for raw, tens in (("q2_dq1", "q2_dq1dq1"), ("p2_dq1", "p2_dq1dq1"), ("q2_dp1", "q2_dq1dp1"), ("p2_dp1", "p2_dq1dp1")):
            fd = (lp[raw] - lm[raw]) / (2 * eps)
            assert np.max(np.abs(fd[0] - out[tens][0, a])) < 2e-6 * max(1.0, np.max(np.abs(fd))), (tens, a)


def test_spline_pendulum_rollout(lib):
    g = G.golden("spline_pendulum")
    s = lib.System(G.desc("spline_pendulum"))
    dt, nsteps, sample = float(g["roll_dt"]), int(g["roll_nsteps"]), int(g["roll_sample"])
    p0 = s.calc_p2(dt, g["roll_q0"], g["roll_q1"])
    G.assert_close(p0[0], g["roll_p_init"], "spline_pendulum p_init")
    out = s.step(g["roll_q1"], p0, dt, dt, nsteps=nsteps, sample_every=sample)
    assert out["status"][0] == 0
    ns = nsteps // sample
    G.assert_close(out["traj_q"][0, :ns], g["roll_q"][1:1 + ns], "spline_pendulum traj q", rtol=1e-7)
    G.assert_close(out["traj_p"][0, :ns], g["roll_p"][1:1 + ns], "spline_pendulum traj p", rtol=1e-7)


def test_pccd_iteration_counts_on_a_large_batch(lib):
    """3000 perturbed points of the pccd rollout through every kernel flavour (table-driven thread kernel,
    cooperative run-time-size and compile-time-size kernels) against the pinned results: same status, results to
    1e-10 and at most a handful of Newton iteration counts differing (against the live reference: none)."""
    rng = np.random.default_rng(21)
    d = G.desc("pccd")
    nq, nd = d.nq, d.nd
    B = 3000
    g = G.golden("pccd")
    idx = rng.integers(1, g["roll_q"].shape[0] - 1, B)
    q1 = g["roll_q"][idx] + rng.normal(0, 0.01, (B, nq)); p1 = g["roll_p"][idx] + rng.normal(0, 0.05, (B, nd))
    lam = g["roll_lambda"][idx - 1]
    u1 = np.zeros((B, 0)); k2 = np.zeros((B, 0)); t1 = np.zeros(B); t2 = t1 + 0.01
    want = G.expected("pccd_large_batch", lambda: G.library_cases("pccd", t1, t2, q1, p1, u1, k2, lambda_guess=lam,
                                                                  deriv1=False))
    for kw in (dict(specialize=False, cooperative=False), dict(specialize=False, cooperative=True), {}):
        s = lib.System(G.desc("pccd"), **kw)
        out = s.linearize(q1, p1, u1, k2, t1=t1, t2=t2, lambda_guess=lam)
        assert np.array_equal(out["status"], want["status"]), s.kernel_name
        ok = want["status"] == 0
        G.assert_cases_close(out, want, ("q2", "p2", "lambda1"), "pccd[%s]" % s.kernel_name)
        assert int(np.sum(out["iters"][ok] != want["iters"][ok])) <= 3, s.kernel_name


def test_device_sincos_accuracy(lib):
    """The kernels' own sin / cos (constant-memory coefficients, trepb_math.cuh sincos_dev) against libm:
    within 2 ulp over the range rollouts visit, exact at 0, library path for huge arguments, NaN for NaN / inf."""
    rng = np.random.default_rng(0)
    x = np.concatenate([rng.uniform(-10, 10, 200000), rng.uniform(-1e5, 1e5, 100000), rng.uniform(-1e-3, 1e-3, 50000),
                        np.array([0.0, -0.0, np.pi / 2, np.pi, -np.pi, 1e5, -1e5, 3e5, 1e12])])
    s, c = lib.sincos(x)
    for got, want in ((s, np.sin(x)), (c, np.cos(x))):
        ulp = np.spacing(np.maximum(np.abs(want), 1e-300))
        err = np.abs(got - want) / ulp
        small = np.abs(want) > 1e-6          # near a zero of sin / cos the absolute error is what matters
        assert np.max(err[small]) <= 2.0, float(np.max(err[small]))
        assert np.max(np.abs(got - want)[~small]) <= 1e-21 + 4e-16 * 1e-6
    assert s[-9] == 0.0 and c[-9] == 1.0
    bad_s, bad_c = lib.sincos(np.array([np.nan, np.inf, -np.inf]))
    assert np.all(np.isnan(bad_s)) and np.all(np.isnan(bad_c))


@pytest.mark.parametrize("name", ["damped_pendulum", "pend_on_cart1", "dual_pendulums"])
def test_iteration_count_flip_rate(lib, name):
    """5000 random single steps per system against the pinned results: how often does a Newton iteration
    count differ?  (The kernels' sin / cos, their division by dt and their convergence test are not the
    reference's instruction sequences; an iterate within rounding distance of the 1e-10 threshold can flip a
    count.  Measured: none in 5000 on every system; the bound leaves room for a handful.)"""
    B, qr, ps, us = 5000, np.pi, 3.0, 2.0
    rng = np.random.default_rng(99)
    d = G.desc(name)
    nq, nd, nu = d.nq, d.nd, d.nu
    q1 = rng.uniform(-qr, qr, (B, nq)); p1 = rng.normal(0, ps, (B, nd)); u1 = rng.uniform(-us, us, (B, nu))
    k2 = np.zeros((B, 0)); t1 = rng.uniform(0, 5, B); t2 = t1 + 0.01
    want = G.expected("flip_rate_" + name, lambda: G.library_cases(name, t1, t2, q1, p1, u1, k2, deriv1=False))
    s = lib.System(G.desc(name))
    out = s.linearize(q1, p1, u1, k2, t1=t1, t2=t2)
    assert np.array_equal(out["status"], want["status"])
    ok = want["status"] == 0
    flips = int(np.sum(out["iters"][ok] != want["iters"][ok]))
    print("%s: %d of %d iteration counts differ" % (name, flips, int(ok.sum())))
    assert flips <= 5
    G.assert_cases_close(out, want, ("q2", "p2"), name)
