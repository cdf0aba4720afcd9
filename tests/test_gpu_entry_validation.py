"""Argument validation of the 24 batch entry points of the C ABI (step, project, linearize, calc_p2, calc_f and
discrete_fm2; plain and _varied; host-pointer and _dev): the exact return code and trepb_last_error() text for each
refused input, and TREPB_OK for a batch of 0.  The C functions are called through lib.raw() so that the Python
wrapper's own checks do not stand in front of them.  The cases without a handle run on the CPU."""
import ctypes as C

import numpy as np
import pytest

import golden_util as G
from test_varied_params import variable_refs
from trep_b200 import desc as D, lib as L

CALLS = ("step", "project", "linearize", "calc_p2", "calc_f", "discrete_fm2")
EVAL = ("calc_p2", "calc_f", "discrete_fm2")
ENTRIES = [(c, v, d) for c in CALLS for v in (False, True) for d in (False, True)]
IDS = ["trepb_%s%s_batch%s" % (c, "_varied" if v else "", "_dev" if d else "") for c, v, d in ENTRIES]
B = 4

INVALID, UNSUPPORTED = 1, 4
NULL = "null argument"
COOP = ("per-instance parameters are not supported by the cooperative kernels (their link tables are built on the "
        "host from the description): create the handle with TREPB_FLAG_NO_COOP")
BATCH = {"step": "batch must be >= 0 and nsteps >= 1", "project": "batch must be >= 0 and nsteps >= 1",
         "linearize": "batch must be >= 0", "calc_p2": "bad batch or dt", "calc_f": "bad batch or t2 == t1",
         "discrete_fm2": "bad batch or t2 == t1"}
DT = {"step": "dt must be non-zero", "project": "dt must be non-zero", "linearize": "dt must be non-zero",
      "calc_p2": "bad batch or dt", "calc_f": "bad batch or t2 == t1", "discrete_fm2": "bad batch or t2 == t1"}
REQUIRED = {"step": ("status", "q1, p1, q2, p2 and status are required"),
            "project": ("status", "bX, bU, Kfb, X, U and status are required"),
            "linearize": ("status", "q1, p1 and status are required"),
            "calc_p2": ("p", NULL), "calc_f": ("f", NULL), "discrete_fm2": ("fm2", NULL)}


def batch_msg(call, dev):
    # the host-pointer evaluations check the batch themselves, before staging
    return "batch must be >= 0" if call in EVAL and not dev else BATCH[call]


def null_varied_msg(call, dev):
    # these _dev entry points check the varied list together with the other pointers
    return NULL if dev and (call == "linearize" or call in EVAL) else "null trepb_varied"


def arrays(d, call, dev, batch=B):
    """Valid arrays of `call` for `batch` instances of d (one step): numpy, or DeviceBuffer for dev."""
    nq, nd, nk, nu, nc = d.nq, d.nd, d.nk, d.nu, d.nc
    nX, nU = 2 * nq, nu + nk
    shapes = {
        "step": dict(q1=(nq,), p1=(nd,), u1=(nu,), k2=(nk,), q2=(nq,), p2=(nd,), lambda1=(nc,), iters=(), status=()),
        "project": dict(bX=(2, nX), bU=(nU,), Kfb=(nU, nX), X=(2, nX), U=(nU,), iters=(), status=()),
        "linearize": dict(q1=(nq,), p1=(nd,), u1=(nu,), k2=(nk,), q2=(nq,), p2=(nd,), lambda1=(nc,), iters=(),
                          status=()),
        "calc_p2": dict(q0=(nq,), q1=(nq,), p=(nd,)),
        "calc_f": dict(q1=(nq,), q2=(nq,), p1=(nd,), f=(nd + nc,)),
        "discrete_fm2": dict(q1=(nq,), q2=(nq,), fm2=(nd,)),
    }[call]
    out = {}
    for k, s in shapes.items():
        shape = (max(batch, 1),) + tuple(max(n, 1) for n in s)
        dtype = np.int32 if k in ("iters", "status") else np.float64
        out[k] = L.DeviceBuffer(0, shape, dtype).zero() if dev else np.zeros(shape, dtype)
    return out


def varied(d, dev, batch=B):
    refs = variable_refs(d)[:1]
    values = np.full((max(batch, 1), 1), getattr(d, D.PAR_TABLE_NAMES[refs[0][0]]).reshape(-1)[refs[0][1]])
    if dev:
        values = L.DeviceBuffer(0, values.shape).upload(values)
    return L._varied((refs, values))


def invoke(h, entry, arr, v, batch=B, dt=0.01, traj_len=0, null_args=False, drop=None):
    call, is_varied, dev = entry
    fn = getattr(L.raw(), "trepb_%s%s_batch%s" % (call, "_varied" if is_varied else "", "_dev" if dev else ""))
    p = {k: (None if null_args or k == drop else L._ptr(x)) for k, x in arr.items()}
    tail = ([C.byref(v) if v is not None else None] if is_varied else []) + ([None] if dev else [])
    if call == "step":
        a = L.StepArgs(batch=batch, nsteps=1, max_iterations=10, t0=0.0, dt=dt, tolerance=1e-10, **p)
    elif call == "project":
        a = L.ProjectArgs(batch=batch, nsteps=1, max_iterations=10, t0=0.0, dt=dt, tolerance=1e-10, use_hint=1, **p)
    elif call == "linearize":
        a = L.LinArgs(batch=batch, max_iterations=10, tolerance=1e-10, t1_scalar=0.0, dt_scalar=dt,
                      traj_len=traj_len, **p)
    if call in ("step", "project", "linearize"):
        args = [None if null_args else C.byref(a)]
    elif call == "calc_p2":
        args = [batch, dt, p["q0"], p["q1"], p["p"]]
    elif call == "calc_f":
        args = [batch, 0.0, dt, p["q1"], p["q2"], p["p1"], None, None, p["f"]]
    else:
        args = [batch, 0.0, dt, p["q1"], p["q2"], None, p["fm2"]]
    rc = fn(h, *args, *tail)
    return rc, (L.raw().trepb_last_error() or b"").decode()


# ---- no handle ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("entry", ENTRIES, ids=IDS)
def test_null_handle(entry):
    d = G.desc("pend_on_cart1")
    v, keep = varied(d, False)
    assert invoke(None, entry, arrays(d, entry[0], False), v) == (INVALID, NULL)


@pytest.mark.parametrize("entry", [e for e in ENTRIES if e[1]], ids=[i for i, e in zip(IDS, ENTRIES) if e[1]])
def test_null_varied_without_handle(entry):
    d = G.desc("pend_on_cart1")
    assert invoke(None, entry, arrays(d, entry[0], False), None) == (INVALID, null_varied_msg(entry[0], entry[2]))


# ---- with a handle --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def handles():
    if L.device_count() < 1:
        pytest.skip("needs a CUDA device")
    return {n: (G.desc(n), L.System(G.desc(n))) for n in ("pend_on_cart1", "damped_pendulum", "puppet")}


def _setup(handles, name, entry, batch=B):
    d, s = handles[name]
    v, keep = varied(d, entry[2], batch)
    return d, s._h, arrays(d, entry[0], entry[2], batch), v, keep


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ENTRIES, ids=IDS)
def test_refusals(handles, entry):
    call, is_varied, dev = entry
    d, h, arr, v, keep = _setup(handles, "pend_on_cart1", entry)
    assert invoke(h, entry, arr, v, null_args=True) == (INVALID, NULL)
    assert invoke(h, entry, arr, v, batch=-1) == (INVALID, batch_msg(call, dev))
    assert invoke(h, entry, arr, v, dt=0.0) == (INVALID, DT[call])
    field, msg = REQUIRED[call]
    assert invoke(h, entry, arr, v, drop=field) == (INVALID, msg)
    if call == "linearize":
        assert invoke(h, entry, arr, v, traj_len=1) == (
            INVALID, "traj_len must be 0 or >= 2 with batch a multiple of traj_len - 1")
    if is_varied:
        assert invoke(h, entry, arr, None) == (INVALID, null_varied_msg(call, dev))
    assert invoke(h, entry, arr, v, batch=0)[0] == 0
    if call == "project":
        d0, h0, arr0, v0, keep0 = _setup(handles, "damped_pendulum", entry)
        assert invoke(h0, entry, arr0, v0) == (INVALID, "the system has no inputs to feed back")


@pytest.mark.gpu
@pytest.mark.parametrize("entry", [e for e in ENTRIES if e[1]], ids=[i for i, e in zip(IDS, ENTRIES) if e[1]])
def test_varied_on_a_cooperative_handle(handles, entry):
    d, h, arr, v, keep = _setup(handles, "puppet", entry)
    assert L.raw().trepb_system_is_cooperative(h)
    assert invoke(h, entry, arr, v) == (UNSUPPORTED, COOP)
    assert invoke(h, entry, arr, v, batch=0)[0] == 0
