"""Argument validation of the tracking-cost and line-search-candidate calls (trepb_track_batch[_dev],
trepb_candidates_batch[_dev]) and the layout of their argument structs.  Every refusal happens before any CUDA call, so
these run without a device: the exact return code and trepb_last_error() text of each refused input, and TREPB_OK for
an empty batch.  Also the host-side pieces of discopt.DOptimizer that need no device."""
import ctypes as C

import numpy as np
import pytest

from test_sweeps import header_struct_size
from trep_b200 import discopt
from trep_b200 import lib as L

INVALID = 1
FAKE = 0x1000          # a non-null address: never dereferenced by a refused call or an empty batch

TRACK_IN = ("X", "U", "Xd", "Ud", "Q", "R", "ref_index", "dX", "dU", "fdxdx", "fdxdu", "fdudu")
TRACK_OUT = ("cost", "dcost", "q", "r", "l_dx", "m_dx", "Qm", "Sm", "Rm")
CAND = ("rows", "lam", "X", "U", "dX", "dU", "Kproj", "bX", "bU", "Kc")
COST_MSG = "X, Xd and Q are required for the cost outputs, and U, Ud and R when nU > 0"
DCOST_MSG = "dcost needs dX and dU"
NEWTON_MSG = "fdxdx, fdxdu and fdudu go together"
MODEL_MSG = "the model needs Qm and Q, and Rm and R when nU > 0"
CAND_MSG = "lam, X, dX and bX are required, and U, dU, Kproj, bU and Kc when nU > 0"
ENTRIES = [("track", False), ("track", True), ("candidates", False), ("candidates", True)]
IDS = ["trepb_%s_batch%s" % (c, "_dev" if d else "") for c, d in ENTRIES]


def track_args(batch=2, nsteps=3, nX=4, nU=1, nref=1, **null):
    a = L.TrackArgs(batch=batch, nsteps=nsteps, nX=nX, nU=nU, nref=nref)
    for f in TRACK_IN + TRACK_OUT:
        setattr(a, f, None if f in null else FAKE)
    return a


def cand_args(groups=2, ncand=8, nsteps=3, nX=4, nU=1, nrollouts=2, **null):
    a = L.CandidatesArgs(groups=groups, ncand=ncand, nsteps=nsteps, nX=nX, nU=nU, nrollouts=nrollouts)
    for f in CAND:
        setattr(a, f, None if f in null else FAKE)
    return a


def args(name, **kw):
    return track_args(**kw) if name == "track" else cand_args(**kw)


def call(name, dev, a):
    fn = getattr(L.raw(), "trepb_%s_batch%s" % (name, "_dev" if dev else ""))
    ptr = None if a is None else C.byref(a)
    return fn(0, ptr, None) if dev else fn(0, ptr)


def expect(rc, code, msg):
    assert rc == code
    if code:
        assert L.raw().trepb_last_error().decode() == msg


@pytest.mark.parametrize("name,dev", ENTRIES, ids=IDS)
def test_null_arguments_are_refused(name, dev):
    expect(call(name, dev, None), INVALID, "null argument")


@pytest.mark.parametrize("dev", [False, True], ids=["host", "dev"])
@pytest.mark.parametrize("sizes", [dict(batch=-1), dict(nsteps=0), dict(nX=0), dict(nU=-1), dict(nref=0),
                                   dict(nsteps=1 << 20, nX=80)],
                         ids=["batch", "nsteps", "nX", "nU", "nref", "model_too_large"])
def test_track_bad_sizes_are_refused(dev, sizes):
    expect(call("track", dev, track_args(**sizes)), INVALID, "bad sizes")


@pytest.mark.parametrize("dev", [False, True], ids=["host", "dev"])
@pytest.mark.parametrize("sizes", [dict(groups=-1), dict(ncand=0), dict(ncand=-3), dict(nsteps=0), dict(nX=0),
                                   dict(nU=-1), dict(nrollouts=-1)],
                         ids=["groups", "M=0", "M<0", "nsteps", "nX", "nU", "nrollouts"])
def test_candidates_bad_sizes_are_refused(dev, sizes):
    expect(call("candidates", dev, cand_args(**sizes)), INVALID, "bad sizes")


@pytest.mark.parametrize("dev", [False, True], ids=["host", "dev"])
def test_track_missing_arrays_are_refused(dev):
    for f in ("X", "U", "Xd", "Ud", "Q", "R"):
        expect(call("track", dev, track_args(**{f: 1})), INVALID, COST_MSG)
    # dcost without the direction
    for f in ("dX", "dU"):
        expect(call("track", dev, track_args(**{f: 1})), INVALID, DCOST_MSG)
    # only some of the three Newton blocks
    for null in (("fdxdx",), ("fdxdu",), ("fdudu",), ("fdxdx", "fdxdu"), ("fdxdu", "fdudu")):
        expect(call("track", dev, track_args(**{f: 1 for f in null})), INVALID, NEWTON_MSG)
    # the model outputs without their weights / each other; the Newton blocks without the model
    model_only = {f: 1 for f in ("X", "U", "Xd", "Ud", "dX", "dU", "cost", "dcost", "q", "r", "l_dx", "m_dx")}
    for f in ("Qm", "Rm", "Q", "R"):
        expect(call("track", dev, track_args(**model_only, **{f: 1})), INVALID, MODEL_MSG)
    expect(call("track", dev, track_args(**model_only, Qm=1, Sm=1, Rm=1)), INVALID, MODEL_MSG)
    expect(call("track", dev, track_args(**{f: 1 for f in TRACK_OUT})), INVALID, MODEL_MSG)


@pytest.mark.parametrize("dev", [False, True], ids=["host", "dev"])
def test_track_optional_arrays_may_be_null(dev):
    # every output optional, no direction without dcost, no Newton blocks, no reference index (empty batch: no run)
    newton = ("fdxdx", "fdxdu", "fdudu")
    for null in (TRACK_OUT + newton, ("dX", "dU", "dcost"), newton, ("ref_index",), ("Qm", "Sm", "Rm") + newton, ("Sm",),
                 ("cost", "dcost", "q", "r", "l_dx", "m_dx", "X", "U", "Xd", "Ud", "dX", "dU")):
        expect(call("track", dev, track_args(batch=0, **{f: 1 for f in null})), 0, "")


@pytest.mark.parametrize("dev", [False, True], ids=["host", "dev"])
def test_candidates_missing_arrays_are_refused(dev):
    for f in ("lam", "X", "dX", "bX", "U", "dU", "Kproj", "bU", "Kc"):
        expect(call("candidates", dev, cand_args(**{f: 1})), INVALID, CAND_MSG)
    expect(call("candidates", dev, cand_args(groups=0, rows=1)), 0, "")


@pytest.mark.parametrize("name,dev", ENTRIES, ids=IDS)
def test_a_system_without_inputs_needs_no_input_arrays(name, dev):
    if name == "track":
        null = ("U", "Ud", "R", "dU", "fdxdu", "fdudu", "r", "Sm", "Rm")
        expect(call(name, dev, track_args(batch=0, nU=0, **{f: 1 for f in null})), 0, "")
        expect(call(name, dev, track_args(nU=0, X=1, **{f: 1 for f in null})), INVALID, COST_MSG)
    else:
        null = ("U", "dU", "Kproj", "bU", "Kc")
        expect(call(name, dev, cand_args(groups=0, nU=0, **{f: 1 for f in null})), 0, "")
        expect(call(name, dev, cand_args(nU=0, X=1, **{f: 1 for f in null})), INVALID, CAND_MSG)


@pytest.mark.parametrize("name,dev", ENTRIES, ids=IDS)
def test_empty_batch_succeeds(name, dev):
    kw = dict(batch=0) if name == "track" else dict(groups=0)
    expect(call(name, dev, args(name, **kw)), 0, "")


def test_ctypes_structs_match_the_header():
    assert C.sizeof(L.TrackArgs) == header_struct_size("trepb_track_args") == 8 + 4 * 4 + 21 * 8
    assert C.sizeof(L.CandidatesArgs) == header_struct_size("trepb_candidates_args") == 8 + 4 * 4 + 8 + 10 * 8
    assert [f for f, _ in L.TrackArgs._fields_] == ["batch", "nsteps", "nX", "nU", "nref"] + list(TRACK_IN + TRACK_OUT)
    assert [f for f, _ in L.CandidatesArgs._fields_] == ["groups", "ncand", "nsteps", "nX", "nU", "nrollouts"] + \
        list(CAND)


def test_the_new_entry_points_are_exported():
    for n in ("trepb_track_batch", "trepb_track_batch_dev", "trepb_candidates_batch", "trepb_candidates_batch_dev"):
        assert n in L.EXPORTS and hasattr(L.raw(), n)


def test_dcost_methods_follow_the_reference_formulas():
    rng = np.random.default_rng(0)
    K, nX, nU = 5, 3, 2
    xd, ud = rng.normal(size=(K + 1, nX)), rng.normal(size=(K, nU))
    Q, R = np.diag([1.0, 2.0, 3.0]), np.array([[2.0, 0.5], [0.5, 1.0]])
    c = discopt.DCost(xd, ud, Q, R)
    x, u = rng.normal(size=nX), rng.normal(size=nU)
    dx, du = x - xd[2], u - ud[2]
    assert np.isclose(c.l(x, u, 2), 0.5 * (dx @ Q @ dx + du @ R @ du))
    assert np.isclose(c.m(x), 0.5 * (x - xd[-1]) @ Q @ (x - xd[-1]))
    assert np.allclose(c.l_dx(x, u, 2), dx @ Q) and np.allclose(c.l_du(x, u, 2), du @ R)
    assert np.allclose(c.m_dx(x), (x - xd[-1]) @ Q)
    assert c.l_dxdx(x, u, 2) is c.Q and c.l_dudu(x, u, 2) is c.R and c.m_dxdx(x) is c.Q
    assert c.l_dxdu(x, u, 2).shape == (nX, nU) and not c.l_dxdu(x, u, 2).any()
    # one reference per rollout: the leading axis runs over the rollouts
    cr = discopt.DCost(np.stack([xd, 2 * xd]), np.stack([ud, ud]), Q, R)
    X = np.stack([x, x])
    assert cr.per_rollout and not c.per_rollout
    assert np.allclose(cr.l_dx(X, np.stack([u, u]), 2), [(x - xd[2]) @ Q, (x - 2 * xd[2]) @ Q])


def test_doptimizer_defaults_and_unsupported_options():
    class FakeDSys:
        pass
    opt = discopt.DOptimizer(FakeDSys(), discopt.DCost(np.zeros((3, 2)), np.zeros((2, 1)), np.eye(2), np.eye(1)))
    assert (opt.armijo_beta, opt.armijo_alpha, opt.armijo_max_iterations, opt.descent_tolerance) == (0.7, 1e-5, 30, 1e-6)
    assert (opt.first_method_iterations, opt.first_method, opt.second_method) == (10, "quasi", "newton")
    assert opt.Qproj is None and opt.Rproj is None and opt.armijo_batch == 8
    opt.optimize_ic = True
    with pytest.raises(ValueError, match="optimize_ic"):
        opt.optimize(np.zeros((3, 2)), np.zeros((2, 1)))
    with pytest.raises(ValueError, match="optimize_ic"):
        opt.calc_descent_direction(np.zeros((3, 2)), np.zeros((2, 1)), "quasi")
    opt.optimize_ic = False
    with pytest.raises(ValueError, match="Invalid descent direction method"):
        opt.calc_descent_direction(np.zeros((3, 2)), np.zeros((2, 1)), "bogus")
