"""Per-instance physical parameters on the cooperative kernels (TREPB_FLAG_COOP_VARIED): every flavour a cooperative
handle can select against cooperative handles built from each row's own description, bit for bit; against the
thread fallback at the parity tolerance; unchanged plain calls; the refusals; and DSystem / DOptimizer on the
marionette with per-rollout rows."""
import copy
import os
import subprocess
import sys

import numpy as np
import pytest

import golden_util as G
from test_gpu_varied_params import _inputs, _same
from test_gpu_varied_deriv2 import _costs, _dsys_calls, _refs

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NROWS = 3


@pytest.fixture(scope="module")
def lib():
    from trep_b200 import lib as L
    if L.device_count() < 1:
        pytest.skip("needs a CUDA device")
    return L


def _sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _rows(d, refs, seed, lo=0.7, hi=1.3):
    base = np.array([d.param_value(r) for r in refs])
    return base * np.random.default_rng(seed).uniform(lo, hi, (NROWS, len(refs)))


def _calls(s, d, x, u, k, Kfb, bX, bU, P, PT, L):
    """step (3 steps, sampled), linearize (one row per instance, raw outputs), linearize over trajectories of L <= 3
    sampled states (one row per trajectory), project, calc_p2, calc_f, discrete_fm2."""
    dt, B = 0.01, x["q1"].shape[0]
    out = {}
    out["step"] = s.step(x["q1"], x["p1"], 0.0, dt, nsteps=u.shape[1], u1=u, k2=k, lambda_guess=x["lam"],
                         sample_every=1, params=P)
    out["lin"] = s.linearize(x["q1"], x["p1"], x["u1"], x["k2"], t1=0.0, t2=dt, q2_guess=x["q2g"],
                             lambda_guess=x["lam"], want_raw=True, params=P)
    R = B // (L - 1)
    tq = np.ascontiguousarray(out["step"]["traj_q"][:R, :L])
    tp = np.ascontiguousarray(out["step"]["traj_p"][:R, :L])
    n = R * (L - 1)
    lt = {"q2": np.zeros((n, d.nq)), "A": np.zeros((n, d.nX, d.nX)), "B": np.zeros((n, d.nX, d.nU)),
          "status": np.zeros(n, np.int32), "iters": np.zeros(n, np.int32)}
    s.linearize_raw(False, n, tq, tp, np.ascontiguousarray(u[:R, :L - 1]) if d.nu else None,
                    np.ascontiguousarray(k[:R, 1:L]) if d.nk else None, lt["status"], t1_scalar=0.0, dt_scalar=dt,
                    q2=lt["q2"], iters=lt["iters"], A=lt["A"], B=lt["B"], traj_len=L, params=PT)
    out["traj"] = lt
    if d.nU:
        out["proj"] = s.project(bX, bU, Kfb, 0.0, dt, params=P)
    q2 = out["lin"]["q2"]
    out["eval"] = {"p2": s.calc_p2(dt, x["q1"], q2, params=P),
                   "f": s.calc_f(0.0, dt, x["q1"], q2, x["p1"], x["u1"], out["lin"]["lambda1"], params=P),
                   "fm2": s.discrete_fm2(0.0, dt, x["q1"], q2, x["u1"], params=P)}
    return out


def _workload(d, g, B, seed):
    rng = np.random.default_rng(seed)
    x = _inputs(d, g, B, rng)
    K = 3
    u = np.repeat(x["u1"][:, None, :], K, axis=1)
    k = x["q1"][:, d.nd:][:, None, :] + 0.01 * np.arange(1, K + 1)[None, :, None]
    bX = np.zeros((B, K + 1, d.nX))
    bX[:, :, :d.nq] = x["q1"][:, None]
    bX[:, :, d.nq:d.nq + d.nd] = x["p1"][:, None]
    bU = np.zeros((B, K, d.nU))
    bU[:, :, :d.nu] = u
    Kfb = rng.normal(0, 0.1, (K, d.nU, d.nX))
    return x, u, k, Kfb, bX, bU


def _pick(a, idx):
    return {kk: (v[idx] if isinstance(v, np.ndarray) else v) for kk, v in a.items()}


# (name, System kwargs): the flavours a cooperative handle selects; fourbar's are the wide instantiations
FLAVOURS = [("puppet", {}), ("puppet", dict(coop_two_warps=True)), ("puppet", dict(coop_one_warp=True)),
            ("puppet", dict(specialize=False)), ("pccd", {}), ("loop3d", {}), ("fourbar", dict(cooperative=True)),
            ("fourbar", dict(cooperative=True, specialize=False))]
IDS = ["puppet_ext", "puppet_pair", "puppet_one_warp", "puppet_rt", "pccd", "loop3d", "fourbar_wide", "fourbar_rt_wide"]


@pytest.mark.parametrize("name,kw", FLAVOURS, ids=IDS)
def test_equal_to_per_row_cooperative_handles(lib, name, kw):
    """Three rows of every variable entry but the frame_se3 ones (+-30 %), spread over a batch larger than one round
    of the persistent grid and ragged against its teams: every call equals, bit for bit, a cooperative handle of the
    same flavour built from the row's own description running the plain entry point."""
    d, g = G.desc(name), G.golden(name)
    refs = _refs(d)
    rows = _rows(d, refs, 5)
    s = lib.System(d, coop_varied=True, **kw)
    assert s.cooperative
    info = s.kernel_info(2)
    teams = info["block"] // 32
    B = 2 * (_sms() * teams) // (1 if teams > 2 else 4) + teams // 2 + 3
    B = min(B, 6000)
    L = 3
    B -= B % (L - 1)
    rid = np.arange(B) % NROWS
    R = B // (L - 1)
    rid_t = np.arange(R) % NROWS
    x, u, k, Kfb, bX, bU = _workload(d, g, B, 7)
    got = _calls(s, d, x, u, k, Kfb, bX, bU, (refs, rows[rid]), (refs, rows[rid_t]), L)
    assert np.mean(got["lin"]["status"] == 0) > 0.5, name
    for j in range(NROWS):
        h = lib.System(d.with_params(refs, rows[j]), **kw)
        assert h.kernel_name == s.kernel_name
        want = _calls(h, d, x, u, k, Kfb, bX, bU, None, None, L)
        sel = np.flatnonzero(rid == j)
        for c in [c for c in ("step", "lin", "proj", "eval") if c in got]:
            _same(_pick(got[c], sel), _pick(want[c], sel), "%s row %d %s" % (name, j, c))
        # trajectory r runs on row rid_t[r]; the per-row handle linearizes every trajectory
        selt = np.flatnonzero(np.repeat(rid_t, L - 1) == j)
        _same(_pick(got["traj"], selt), _pick(want["traj"], selt), "%s row %d trajectories" % (name, j))
        h.close()


def test_dev_entry_points_give_the_host_bits(lib):
    """trepb_linearize_varied_batch_dev and trepb_step_varied_batch_dev with device rows, on the marionette."""
    d, g = G.desc("puppet"), G.golden("puppet")
    refs = _refs(d)
    rows = _rows(d, refs, 9)
    s = lib.System(d, coop_varied=True)
    B = 301
    x = _inputs(d, g, B, np.random.default_rng(2))
    vals = np.ascontiguousarray(rows[np.arange(B) % NROWS])
    want = s.linearize(x["q1"], x["p1"], x["u1"], x["k2"], t1=0.0, t2=0.01, want_raw=False, params=(refs, vals))
    dv = lambda a: lib.DeviceBuffer(0, a.shape, a.dtype).upload(np.ascontiguousarray(a))
    st, q2, A = dv(np.zeros(B, np.int32)), dv(np.zeros((B, d.nq))), dv(np.zeros((B, d.nX, d.nX)))
    s.linearize_raw(True, B, dv(x["q1"]), dv(x["p1"]), dv(x["u1"]), dv(x["k2"]), st, t1_scalar=0.0, dt_scalar=0.01,
                    q2=q2, A=A, params=(refs, dv(vals)))
    assert st.download().tobytes() == want["status"].tobytes()
    assert q2.download().tobytes() == want["q2"].tobytes() and A.download().tobytes() == want["A"].tobytes()


def test_against_the_thread_fallback(lib):
    """The same rows (+-5 %) on a TREPB_FLAG_NO_COOP handle (the table-driven thread kernels): equal statuses of
    step and linearize, and the results of the instances both paths converged within the project's parity tolerance
    (iteration counts may differ by one where a residual sits at the tolerance)."""
    d, g = G.desc("puppet"), G.golden("puppet")
    refs = _refs(d)
    rows = _rows(d, refs, 4, 0.95, 1.05)
    B = 96
    x, u, k, Kfb, bX, bU = _workload(d, g, B, 8)
    P = (refs, rows[np.arange(B) % NROWS])
    PT = (refs, rows[np.arange(B // 2) % NROWS])
    a = _calls(lib.System(d, coop_varied=True), d, x, u, k, Kfb, bX, bU, P, PT, 3)
    b = _calls(lib.System(d, cooperative=False), d, x, u, k, Kfb, bX, bU, P, PT, 3)
    for c in a:
        ok = (a[c] if "status" in a[c] else a["lin"])["status"] == 0   # eval runs on the linearize call's q2
        if c in ("step", "lin"):
            assert np.mean(ok) > 0.9 and np.array_equal(a[c]["status"], b[c]["status"]), c
        ok = ok & ((b[c] if "status" in b[c] else b["lin"])["status"] == 0)
        for kk, v in a[c].items():
            if isinstance(v, np.ndarray) and kk not in ("status", "iters", "fail_step"):
                # f is a residual, ~0 at the converged q2: its error is set by the momentum-sized terms it cancels
                scale = max(1.0, float(np.max(np.abs(x["p1"])))) if kk == "f" else None
                G.assert_close(v[ok], b[c][kk][ok], "%s %s" % (c, kk), rtol=1e-10, scale=scale)


def test_base_rows_and_the_flag_change_nothing(lib):
    """A flagged handle selects the same kernels with the same geometry and gives the same bits on plain calls as
    an unflagged one; rows equal to the description's values give the plain call's bits."""
    d, g = G.desc("puppet"), G.golden("puppet")
    refs = _refs(d)
    for kw in ({}, dict(coop_two_warps=True)):
        a, b = lib.System(d, **kw), lib.System(d, coop_varied=True, **kw)
        assert a.kernel_name == b.kernel_name
        for w in range(4):
            assert a.kernel_info(w) == b.kernel_info(w)
        B = 2 * _sms() * 16 + 5
        x, u, k, Kfb, bX, bU = _workload(d, g, B, 3)
        L = 3
        B2 = B - B % (L - 1)
        x = {kk: v[:B2] for kk, v in x.items()}
        u, k, bX, bU = u[:B2], k[:B2], bX[:B2], bU[:B2]
        pa = _calls(a, d, x, u, k, Kfb, bX, bU, None, None, L)
        pb = _calls(b, d, x, u, k, Kfb, bX, bU, None, None, L)
        base = np.array([d.param_value(r) for r in refs])
        vb = _calls(b, d, x, u, k, Kfb, bX, bU, (refs, np.tile(base, (B2, 1))), (refs, np.tile(base, (B2 // 2, 1))), L)
        for c in pa:
            _same(pa[c], pb[c], "flag %s" % c)
            _same(pa[c], vb[c], "base rows %s" % c)


def test_second_derivatives(lib):
    """trepb_deriv2_varied_batch on a flagged cooperative handle (linearize on the varied cooperative kernel, pass A
    on the table-driven map): z-contracted and full tensors equal per-row handles bit for bit."""
    d, g = G.desc("puppet"), G.golden("puppet")
    refs = _refs(d)
    rows = _rows(d, refs, 6, 0.9, 1.1)
    B = 40
    x = _inputs(d, g, B, np.random.default_rng(5))
    rid = np.arange(B) % NROWS
    z = np.random.default_rng(6).normal(0, 1, (B, d.nX))
    s = lib.System(d, coop_varied=True)
    kw = dict(t1=0.0, t2=0.01, q2_guess=x["q2g"], lambda_guess=x["lam"])
    got_z = s.deriv2(x["q1"], x["p1"], x["u1"], x["k2"], z=z, tensors=False, params=(refs, rows[rid]), **kw)
    got_t = s.deriv2(x["q1"], x["p1"], x["u1"], x["k2"], params=(refs, rows[rid]), **kw)
    assert np.mean(got_t["status"] == 0) > 0.5
    for j in range(NROWS):
        h = lib.System(d.with_params(refs, rows[j]))
        sel = np.flatnonzero(rid == j)
        _same(_pick(got_z, sel), _pick(h.deriv2(x["q1"], x["p1"], x["u1"], x["k2"], z=z, tensors=False, **kw), sel),
              "deriv2 z row %d" % j)
        _same(_pick(got_t, sel), _pick(h.deriv2(x["q1"], x["p1"], x["u1"], x["k2"], **kw), sel), "deriv2 row %d" % j)


def test_varied_constant_rotation_angle(lib):
    """A marionette tilted by a constant rotation frame, its angle varied per row.  cos / sin come from the device
    math library here and from the C library in a per-row handle's blob; they may differ by up to 2 ulp, a relative
    change of 4.4e-16 in a few pre-transform entries.  Propagated through a solve whose condition is far below
    1e5, that stays below the parity tolerance of 1e-10 used here; statuses and iteration counts must agree."""
    from trep_b200 import desc as D
    d0, g = G.desc("puppet"), G.golden("puppet")
    d = copy.deepcopy(d0)
    f = [i for i in range(len(d.frame_kind)) if d.frame_config[i] < 0 and D.RX <= d.frame_kind[i] <= D.RZ][0]
    d.frame_value[f] = 0.05
    refs = [(D.PAR_TABLES["frame_value"], f), d.param_ref("pot_d", 0, 2)]
    rows = np.array([[0.05, -9.8], [0.0731, -9.6], [-0.0417, -10.1]])
    B = 60
    x, u, k, Kfb, bX, bU = _workload(d, g, B, 12)
    rid = np.arange(B) % NROWS
    got = _calls(lib.System(d, coop_varied=True), d, x, u, k, Kfb, bX, bU, (refs, rows[rid]), (refs, rows[rid[:30]]), 3)
    rid_t = np.repeat(rid[:30], 2)
    for j in range(NROWS):
        want = _calls(lib.System(d.with_params(refs, rows[j])), d, x, u, k, Kfb, bX, bU, None, None, 3)
        for c in got:
            sel = np.flatnonzero((rid_t if c == "traj" else rid) == j)
            _same(_pick(got[c], sel), _pick(want[c], sel), "angle row %d %s" % (j, c), exact=False)


def test_one_failing_instance(lib):
    """A row that makes one instance's solve fail (a NaN mass) reports a status for that instance only; every
    other instance keeps its bits."""
    d, g = G.desc("puppet"), G.golden("puppet")
    refs = _refs(d)
    rows = _rows(d, refs, 13)
    B = 50
    x = _inputs(d, g, B, np.random.default_rng(1))
    vals = rows[np.arange(B) % NROWS].copy()
    s = lib.System(d, coop_varied=True)
    a = s.linearize(x["q1"], x["p1"], x["u1"], x["k2"], t1=0.0, t2=0.01, want_raw=True, params=(refs, vals))
    m = [i for i, r in enumerate(refs) if r[0] == 2][0]
    vals[17, m] = np.nan
    b = s.linearize(x["q1"], x["p1"], x["u1"], x["k2"], t1=0.0, t2=0.01, want_raw=True, params=(refs, vals))
    assert a["status"][17] == 0 and b["status"][17] != 0
    keep = np.arange(B) != 17
    _same(_pick(a, keep), _pick(b, keep), "other instances")


def test_refusals(lib):
    """Without the flag a cooperative handle refuses as before; with it, entries are checked as on the thread path."""
    d = G.desc("puppet")
    q, p, k2 = np.zeros((4, d.nq)), np.zeros((4, d.nd)), np.zeros((4, 1, d.nk))
    plain = lib.System(d)
    with pytest.raises(lib.TrepbError) as e:
        plain.step(q, p, 0.0, 0.01, k2=k2, params=([d.param_ref("pot_d", 0, 2)], np.full((4, 1), -9.8)))
    assert e.value.code == 4 and "create the handle with TREPB_FLAG_NO_COOP" in str(e.value)
    s = lib.System(d, coop_varied=True)
    zero = [r for r in [(2, 4 * f + 1) for f in range(len(d.frame_kind))] if d.param_value(r) == 0.0][0]
    for refs, pattern in (([zero], r"value is 0"),
                          ([d.param_ref("pot_d", 0, 2)] * 2, r"more than once")):
        with pytest.raises(lib.TrepbError) as e:
            s.step(q, p, 0.0, 0.01, k2=k2, params=(refs, np.ones((4, len(refs)))))
        assert e.value.code == 1 and pattern in str(e.value)
    from trep_b200.lib import _varied
    import ctypes as C
    v, keep = _varied(([d.param_ref("pot_d", 0, 2)], None))
    out = {"status": np.zeros(4, np.int32)}
    a = s._lin_args(4, q, p, None, np.zeros((4, d.nk)), out["status"], t1_scalar=0.0, dt_scalar=0.01)
    rc = lib._lib.trepb_linearize_varied_batch(s._h, C.byref(a), C.byref(v))
    assert rc == 1 and "values is required" in lib._lib.trepb_last_error().decode()


def test_dsystem_and_doptimizer_on_the_marionette(lib):
    """DSystem on the marionette with 8 per-rollout rows: linearize_trajectory, calc_feedback_controller,
    calc_newton_model, project, simulate and f equal one DSystem per rollout bit for bit, and so do
    calc_descent_direction and DOptimizer.step with steepest, quasi and newton."""
    from test_gpu_doptimizer import _problem
    from trep_b200 import discopt, midpointvi as MV
    d, t, _, X, U, cost = _problem("puppet", 8, 6, 21)
    refs = _refs(d)
    vals = np.array([d.param_value(r) for r in refs]) * np.random.default_rng(22).uniform(0.95, 1.05, (8, len(refs)))
    ds = discopt.DSystem(MV.MidpointVI(d), t)
    assert ds.varint.sys.cooperative
    ds.set_parameters(refs, vals)
    X = ds.simulate(X[:, 0], U)
    costs = _costs(ds, 8, 6, 1)
    got = _dsys_calls(ds, X, U, costs)
    opt = discopt.DOptimizer(ds, cost)
    steps = {m: opt.step(0, X, U, m) for m in ("steepest", "quasi", "newton")}
    for r in range(8):
        one = discopt.DSystem(MV.MidpointVI(d.with_params(refs, vals[r])), t)
        w = _dsys_calls(one, X[r:r + 1], U[r:r + 1], [c[r:r + 1] for c in costs])
        for kk in w:
            assert got[kk][r:r + 1].tobytes() == w[kk].tobytes(), "rollout %d %s" % (r, kk)
        o1 = discopt.DOptimizer(one, discopt.DCost(cost.xd[r:r + 1], cost.ud[r:r + 1], cost.Q, cost.R))
        for m, st in steps.items():
            w = o1.step(0, X[r:r + 1], U[r:r + 1], m)
            assert st.X[r].tobytes() == w.X[0].tobytes() and st.U[r].tobytes() == w.U[0].tobytes(), (m, r)
            assert st.cost[r] == w.cost[0] and st.dcost[r] == w.dcost[0], (m, r)


def test_cooperative_plugin(lib):
    """kind="coop" plug-in (the rod's shape): its kernel set carries the varied launchers."""
    code = "import test_gpu_varied_coop as t; t._plugin_check()"
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([HERE, ROOT]))
    r = subprocess.run([sys.executable, "-c", code], cwd=HERE, env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def _plugin_check():
    import shutil
    from trep_b200 import build, lib as L
    d, g = G.desc("rod"), G.golden("rod")
    path = os.path.join(os.path.dirname(build.LIB), "libtrepb_plugin_rod_coop.so")
    if shutil.which(build.NVCC) is not None:
        path = build.build_plugin(d, "rod_coop", kind="coop")
    assert L.load_plugin(path) == 1
    refs = _refs(d)
    rows = _rows(d, refs, 31, 0.9, 1.1)
    s = L.System(d, cooperative=True, coop_varied=True)
    assert s.kernel_name == "cooperative/rod_coop"
    B = 30
    x = _inputs(d, g, B, np.random.default_rng(4))
    rid = np.arange(B) % NROWS
    got = s.linearize(x["q1"], x["p1"], x["u1"], x["k2"], t1=0.0, t2=0.01, want_raw=True, params=(refs, rows[rid]))
    assert np.mean(got["status"] == 0) > 0.5
    for j in range(NROWS):
        h = L.System(d.with_params(refs, rows[j]), cooperative=True)
        sel = np.flatnonzero(rid == j)
        _same(_pick(got, sel), _pick(h.linearize(x["q1"], x["p1"], x["u1"], x["k2"], t1=0.0, t2=0.01, want_raw=True), sel),
              "plug-in row %d" % j)
