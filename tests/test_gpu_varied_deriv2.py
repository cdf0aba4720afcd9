"""Per-instance physical parameters for second derivatives (trepb_deriv2_varied_batch*) and for DSystem's
trajectory-optimisation calls (DSystem.set_parameters): anchored to the reference's goldens, equal to handles built
from each instance's own description, unchanged without variation, and the refusals.  The cases without a handle run
on the CPU."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import golden_util as G
from test_gpu_varied_params import NOT_BITWISE, SYSTEMS, _inputs, _same
from test_varied_params import variable_refs
from trep_b200 import lib as L

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
INVALID, UNSUPPORTED = 1, 4

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    if L.device_count() < 1:
        pytest.skip("needs a CUDA device")
    return L


def _refs(d):
    return [r for r in variable_refs(d) if r[0] != 1]


# ---- 1. anchored to the reference ---------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name,kw", [("pend_on_cart1", {}), ("fourbar", dict(specialize=False, cooperative=False)),
                                     ("fourbar", dict(specialize=False, cooperative=False, d2_pairwise=True))],
                         ids=["pend_on_cart1", "fourbar_d2jac", "fourbar_pairwise"])
def test_anchored_to_the_reference(lib, name, kw):
    """The handle is built from the same structure with every variable entry scaled by 1.25; rows carrying the
    golden description's own numbers reproduce the reference's 30 tensors."""
    d, g = G.desc(name), G.golden(name)
    refs = _refs(d)
    base = np.array([d.param_value(r) for r in refs])
    s = lib.System(d.with_params(refs, 1.25 * base), **kw)
    n = len(g["case_iters"])
    kwargs = dict(t1=g["case_t1"], t2=g["case_t2"], q2_guess=g["case_q2_guess"], lambda_guess=g["case_lambda_guess"])
    out = s.deriv2(g["case_q1"], g["case_p1"], g["case_u1"], g["case_k2"], params=(refs, np.tile(base, (n, 1))), **kwargs)
    ref = lib.System(d, **kw).deriv2(g["case_q1"], g["case_p1"], g["case_u1"], g["case_k2"], **kwargs)
    assert np.all(out["status"] == 0)
    assert np.array_equal(out["status"], ref["status"]) and np.array_equal(out["iters"], ref["iters"])
    assert np.array_equal(out["iters"], g["case_iters"])
    G.assert_close(out["A"], g["case_A"], name + " A")
    G.assert_d2_close(out, g, name)


# ---- 2. equal to per-instance handles -----------------------------------------------------------------------------
D2_SYSTEMS = [(n, kw) for n, kw in SYSTEMS if n != "puppet"] + [("rod", dict(specialize=False, cooperative=False,
                                                                              d2_pairwise=True))]


def _d2_case(d, g, B, seed):
    rng = np.random.default_rng(seed)
    refs = _refs(d)
    vals = np.array([d.param_value(r) for r in refs]) * rng.uniform(0.5, 1.5, (B, len(refs)))
    x = _inputs(d, g, B, rng)
    z = rng.normal(0, 1, (B, d.nX))
    return refs, vals, x, z


def _deriv2(h, x, z, sl, params=None, dt=0.01):
    one = lambda a: a[sl]
    return h.deriv2(one(x["q1"]), one(x["p1"]), one(x["u1"]), one(x["k2"]), t1=0.0, t2=dt, q2_guess=one(x["q2g"]),
                    lambda_guess=one(x["lam"]), z=one(z), params=params)


@gpu
@pytest.mark.parametrize("name,kw", D2_SYSTEMS, ids=[n + ("_pairwise" if kw.get("d2_pairwise") else "")
                                                     for n, kw in D2_SYSTEMS])
def test_equal_to_per_instance_handles(lib, name, kw):
    """64 instances, every variable entry drawn +-50 % around the base: deriv2 (all 30 tensors, the deriv1 arrays and
    the z-contracted fdxdx / fdxdu / fdudu) against a handle built from that instance's own description running the
    plain entry point.  pend_on_cart1 from its golden description runs on the all-literal instantiation, so its
    varied call switches to the run-time-parameter kernels of the structure."""
    d, g = G.desc(name), G.golden(name)
    B = 64
    refs, vals, x, z = _d2_case(d, g, B, 21)
    s = lib.System(d, **kw)
    assert s.specialized == ("specialize" not in kw) and not s.cooperative
    got = _deriv2(s, x, z, slice(None), params=(refs, vals))
    assert np.mean(got["status"] == 0) > 0.5, name
    ex = name not in NOT_BITWISE
    for b in range(B):
        h = lib.System(d.with_params(refs, vals[b]), **kw)
        w = _deriv2(h, x, z, slice(b, b + 1))
        _same({k: v[b:b + 1] for k, v in got.items()}, w, "%s deriv2 %d" % (name, b), ex)
        h.close()


@gpu
def test_plugin_matches_per_instance_handles(lib):
    """A structure specialised at run time (lib.specialize), in a fresh interpreter: plug-ins stay registered for the
    life of a process."""
    code = "import test_gpu_varied_deriv2 as t; t._plugin_check()"
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(filter(None, [ROOT, HERE, os.environ.get("PYTHONPATH")])))
    subprocess.run([sys.executable, "-c", code], cwd=HERE, env=env, check=True)


def _plugin_check():
    d, g = G.desc("damper_only"), G.golden("damper_only")
    L.specialize(d)
    s = L.System(d)
    assert s.specialized
    B = 64
    refs, vals, x, z = _d2_case(d, g, B, 5)
    got = _deriv2(s, x, z, slice(None), params=(refs, vals))
    assert np.mean(got["status"] == 0) > 0.5
    for b in range(B):
        h = L.System(d.with_params(refs, vals[b]))
        assert h.specialized
        _same({k: v[b:b + 1] for k, v in got.items()}, _deriv2(h, x, z, slice(b, b + 1)), "plug-in %d" % b)
        h.close()


# ---- 3. no variation means no change ------------------------------------------------------------------------------
def _deriv2_dev(s, d, x, z, B, params=None, dt=0.01):
    """The _dev entry point on DeviceBuffers: q2, status, iters, three tensors and the z-contractions."""
    up = lambda a, dtype=np.float64: L.DeviceBuffer(0, a.shape, dtype).upload(np.ascontiguousarray(a, dtype=dtype))
    ins = dict(q1=up(x["q1"]), p1=up(x["p1"]), u1=up(x["u1"]) if d.nu else None, k2=up(x["k2"]) if d.nk else None,
               t1=up(np.zeros(B)), t2=up(np.full(B, dt)), q2g=up(x["q2g"]), z=up(z))
    shapes = s.d2_shapes(B)
    names = ["q2_dq1dq1", "p2_dq1dp1", "q2_dp1dp1"]
    outs = dict(q2=(B, d.nq), status=(B,), iters=(B,), fdxdx=(B, d.nX, d.nX), **{n: shapes[n] for n in names})
    if d.nU:
        outs.update(fdxdu=(B, d.nX, d.nU), fdudu=(B, d.nU, d.nU))
    ob = {k: L.DeviceBuffer(0, sh, np.int32 if k in ("status", "iters") else np.float64).zero() for k, sh in outs.items()}
    dpar = None if params is None else (params[0], up(params[1]))
    s.deriv2_raw(True, B, ins["q1"], ins["p1"], ins["u1"], ins["k2"], ob["status"], {n: ob[n] for n in names},
                 z=ins["z"], fdxdx=ob["fdxdx"], fdxdu=ob.get("fdxdu"), fdudu=ob.get("fdudu"), t1=ins["t1"],
                 t2=ins["t2"], q2_guess=ins["q2g"], q2=ob["q2"], iters=ob["iters"], params=dpar)
    L.synchronize(0)
    return {k: v.download() for k, v in ob.items()}


@gpu
@pytest.mark.parametrize("name,kw", [("pend_on_cart2", dict(literal=False)),
                                     ("fourbar", dict(specialize=False, cooperative=False)),
                                     ("rod", dict(specialize=False, cooperative=False, d2_pairwise=True))],
                         ids=["pend_on_cart2", "fourbar_d2jac", "rod_pairwise"])
def test_no_variation_means_no_change(lib, name, kw):
    """Rows equal to the description's values: the same bits as the plain deriv2 of the same handle, host-pointer and
    _dev forms."""
    d, g = G.desc(name), G.golden(name)
    B = 300
    refs, _, x, z = _d2_case(d, g, B, 8)
    P = (refs, np.tile([d.param_value(r) for r in refs], (B, 1)))
    s = lib.System(d, **kw)
    _same(_deriv2(s, x, z, slice(None)), _deriv2(s, x, z, slice(None), params=P), name + " host")
    _same(_deriv2_dev(s, d, x, z, B), _deriv2_dev(s, d, x, z, B, params=P), name + " dev")


# ---- 4. refusals --------------------------------------------------------------------------------------------------
def _raw(h, dev, v, batch=4, traj_len=0):
    fn = getattr(L.raw(), "trepb_deriv2_varied_batch%s" % ("_dev" if dev else ""))
    a = L.D2Args()
    a.lin = L.LinArgs(batch=batch, max_iterations=10, tolerance=1e-10, t1_scalar=0.0, dt_scalar=0.01, traj_len=traj_len)
    rc = fn(h, C.byref(a), C.byref(v) if v is not None else None, *([None] if dev else []))
    return rc, (L.raw().trepb_last_error() or b"").decode()


@pytest.mark.parametrize("dev", [False, True], ids=["host", "dev"])
def test_refusals_without_handle(dev):
    d = G.desc("pend_on_cart1")
    refs = variable_refs(d)[:1]
    v, keep = L._varied((refs, np.full((4, 1), d.param_value(refs[0]))))
    assert _raw(None, dev, v) == (INVALID, "null argument")
    assert _raw(None, dev, None) == (INVALID, "null trepb_varied")


@gpu
def test_refusals(lib):
    p = G.desc("pend_on_cart1")
    sp = lib.System(p)
    zeros = lambda n: np.zeros((4, n))
    with pytest.raises(lib.TrepbError) as e:   # a structural entry
        sp.deriv2(zeros(p.nq), zeros(p.nd), zeros(p.nu), t1=0.0, t2=0.01,
                  params=([p.param_ref("pot_d", 0, 0)], np.ones((4, 1))))
    assert e.value.code == INVALID and "POT_D[0]" in str(e.value)
    refs = variable_refs(p)[:1]
    for dev in (False, True):
        vals = np.full((4, 1), p.param_value(refs[0]))
        v, keep = L._varied((refs, L.DeviceBuffer(0, vals.shape).upload(vals) if dev else vals))
        assert _raw(sp._h, dev, v, traj_len=3) == (
            INVALID, "per-instance parameters of second derivatives take one row per instance: traj_len must be 0")
        assert _raw(sp._h, dev, None) == (INVALID, "null trepb_varied")
        assert _raw(sp._h, dev, v, batch=0)[0] == 0
    d = G.desc("puppet")
    s = lib.System(d)
    assert s.cooperative
    with pytest.raises(lib.TrepbError) as e:
        s.deriv2(np.zeros((4, d.nq)), np.zeros((4, d.nd)), k2=np.zeros((4, d.nk)), t1=0.0, t2=0.01,
                 params=([d.param_ref("pot_d", 0, 2)], np.full((4, 1), -9.8)))
    assert e.value.code == UNSUPPORTED and "TREPB_FLAG_NO_COOP" in str(e.value)


# ---- 5. DSystem ---------------------------------------------------------------------------------------------------
def _dsys(d, specialize, t):
    from trep_b200 import discopt, midpointvi as MV
    return discopt.DSystem(MV.MidpointVI(d, specialize=specialize), t)


def _traj(d, g, R, K, rng):
    x = _inputs(d, g, R, rng)
    X = np.zeros((R, K + 1, d.nX))
    X[:, :, :d.nq] = x["q1"][:, None] + 0.002 * np.arange(K + 1)[None, :, None]
    X[:, :, d.nq:d.nq + d.nd] = x["p1"][:, None]
    U = np.zeros((R, K, d.nU))
    U[:, :, :d.nu] = x["u1"][:, None]
    U[:, :, d.nu:] = X[:, 1:, d.nq - d.nk:d.nq]
    return X, U


def _costs(ds, R, K, seed):
    """Cost gradients l_dx [R,K,nX], l_du [R,K,nU], m_dx [R,nX] of the newton model."""
    rng = np.random.default_rng(seed)
    return rng.normal(0, 1, (R, K, ds.nX)), rng.normal(0, 1, (R, K, ds.nU)), rng.normal(0, 1, (R, ds.nX))


def _dsys_calls(ds, X, U, costs):
    """linearize_trajectory, calc_newton_model, calc_feedback_controller, project, simulate and f on (X, U)."""
    out = {}
    A, B = ds.linearize_trajectory(X, U)
    out.update(A=A, B=B)
    Kfb, A2, B2 = ds.calc_feedback_controller(X, U, return_linearization=True)
    out.update(Kfb=Kfb, A2=A2, B2=B2)
    for k, v in zip(("z", "fxx", "fxu", "fuu"), ds.calc_newton_model(X, U, A, B, Kfb, *costs)):
        out[k] = v
    out["Xp"], out["Up"] = ds.project(X, U, Kfb)
    out["Xs"] = ds.simulate(X[:, 0], U)
    out["f"] = ds.f(X[:, 0], U[:, 0], 0)
    return out


@gpu
@pytest.mark.parametrize("name,specialize", [("pend_on_cart1", True), ("pend_on_cart2", False)],
                         ids=["pend_on_cart1", "pend_on_cart2_table"])
def test_dsystem_rollouts(lib, name, specialize):
    """R = 8 rollouts, each on its own parameter row, against one DSystem per rollout built on that row's description:
    bitwise equal.  A single row broadcasts; a row count that fits neither rollouts nor instances raises; without
    set_parameters nothing changes."""
    d, g = G.desc(name), G.golden(name)
    R, K = 8, 6
    t = np.arange(K + 1) * 0.01
    rng = np.random.default_rng(13)
    refs = _refs(d)
    base = np.array([d.param_value(r) for r in refs])
    vals = base * rng.uniform(0.8, 1.2, (R, len(refs)))
    X, U = _traj(d, g, R, K, rng)
    ds = _dsys(d, specialize, t)
    costs = _costs(ds, R, K, 1)
    plain = _dsys_calls(ds, X, U, costs)
    ds.set_parameters(refs, vals)
    got = _dsys_calls(ds, X, U, costs)
    for r in range(R):
        one = _dsys(d.with_params(refs, vals[r]), specialize, t)
        w = _dsys_calls(one, X[r:r + 1], U[r:r + 1], [c[r:r + 1] for c in costs])
        for k in w:
            assert got[k][r:r + 1].tobytes() == w[k].tobytes(), "%s rollout %d %s" % (name, r, k)
    # one row for every rollout
    ds.set_parameters(refs, base * 1.1)
    one = _dsys(d.with_params(refs, base * 1.1), specialize, t)
    a, b = _dsys_calls(ds, X, U, costs), _dsys_calls(one, X, U, costs)
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), "%s single row %s" % (name, k)
    # rows that fit neither the rollouts nor the instances
    ds.set_parameters(refs, vals[:3])
    with pytest.raises(ValueError):
        ds.linearize_trajectory(X, U)
    with pytest.raises(ValueError):
        ds.f(X[:, 0], U[:, 0], 0)
    # parameters on both the DSystem and its MidpointVI
    ds.set_parameters(refs, vals)
    ds.varint.set_parameters(refs, vals)
    with pytest.raises(ValueError):
        ds.simulate(X[:, 0], U)
    ds.varint.set_parameters(None, None)
    # cleared: the results of a DSystem that never had parameters
    ds.set_parameters(None, None)
    again = _dsys_calls(ds, X, U, costs)
    for k in plain:
        assert again[k].tobytes() == plain[k].tobytes(), "%s cleared %s" % (name, k)
