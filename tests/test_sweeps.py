"""Argument validation of the tangent and adjoint sweeps (trepb_tangent_batch[_dev], trepb_adjoint_batch[_dev]) and
the layout of their argument structs.  Every refusal happens before any CUDA call, so these run without a device:
the exact return code and trepb_last_error() text of each refused input, and TREPB_OK for a batch of 0."""
import ctypes as C
import os
import re

import pytest

from trep_b200 import lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID = 1
FAKE = 0x1000          # a non-null address: never dereferenced by a refused call or a batch of 0

TANGENT_MSG = "A and dX are required, and B, K and dU when nU > 0"
ADJOINT_MSG = "A, m_dx and z are required, and B when K is given"
ENTRIES = [("tangent", False), ("tangent", True), ("adjoint", False), ("adjoint", True)]
IDS = ["trepb_%s_batch%s" % (c, "_dev" if d else "") for c, d in ENTRIES]


def full_args(call, batch=2, nsteps=3, nX=4, nU=1, **null):
    """Arguments with every array present (fake addresses), then the fields named in `null` set to NULL."""
    if call == "tangent":
        a = L.TangentArgs(batch=batch, nsteps=nsteps, nX=nX, nU=nU)
        fields = ("A", "B", "K", "bdX", "bdU", "x0", "dX", "dU")
    else:
        a = L.AdjointArgs(batch=batch, nsteps=nsteps, nX=nX, nU=nU)
        fields = ("A", "B", "K", "l_dx", "l_du", "m_dx", "z", "z1")
    for f in fields:
        setattr(a, f, None if f in null else FAKE)
    return a


def call(name, dev, args):
    fn = getattr(L.raw(), "trepb_%s_batch%s" % (name, "_dev" if dev else ""))
    ptr = None if args is None else C.byref(args)
    return fn(0, ptr, None) if dev else fn(0, ptr)


def expect(rc, code, msg):
    assert rc == code
    if code:
        assert L.raw().trepb_last_error().decode() == msg


@pytest.mark.parametrize("name,dev", ENTRIES, ids=IDS)
def test_null_arguments_are_refused(name, dev):
    expect(call(name, dev, None), INVALID, "null argument")


@pytest.mark.parametrize("name,dev", ENTRIES, ids=IDS)
@pytest.mark.parametrize("sizes", [dict(batch=-1), dict(nsteps=0), dict(nX=0), dict(nU=-1)],
                         ids=["batch", "nsteps", "nX", "nU"])
def test_bad_sizes_are_refused(name, dev, sizes):
    expect(call(name, dev, full_args(name, **sizes)), INVALID, "bad sizes")


@pytest.mark.parametrize("name,dev", ENTRIES, ids=IDS)
def test_missing_arrays_are_refused(name, dev):
    if name == "tangent":
        missing, optional = ("A", "B", "K", "dX", "dU"), ("bdX", "bdU", "x0")
        msg = TANGENT_MSG
    else:
        missing, optional = ("A", "m_dx", "z"), ("K", "l_dx", "l_du", "z1")
        msg = ADJOINT_MSG
    for f in missing:
        expect(call(name, dev, full_args(name, **{f: 1})), INVALID, msg)
    # the optional arrays may all be NULL (checked with a batch of 0: nothing runs)
    expect(call(name, dev, full_args(name, batch=0, **{f: 1 for f in optional})), 0, "")
    if name == "adjoint":
        # B is needed only with K: the open-loop costate reads A alone
        expect(call(name, dev, full_args(name, B=1)), INVALID, msg)
        expect(call(name, dev, full_args(name, batch=0, B=1, K=1)), 0, "")


@pytest.mark.parametrize("name,dev", ENTRIES, ids=IDS)
def test_a_system_without_inputs_needs_no_input_arrays(name, dev):
    # nU == 0: B, K, bdU / l_du and dU may be NULL; a size check still applies to the rest
    null = ("B", "K", "bdU", "dU") if name == "tangent" else ("B", "K", "l_du")
    expect(call(name, dev, full_args(name, batch=0, nU=0, **{f: 1 for f in null})), 0, "")
    expect(call(name, dev, full_args(name, nU=0, A=1, **{f: 1 for f in null})), INVALID,
           TANGENT_MSG if name == "tangent" else ADJOINT_MSG)


@pytest.mark.parametrize("name,dev", ENTRIES, ids=IDS)
def test_empty_batch_succeeds(name, dev):
    expect(call(name, dev, full_args(name, batch=0)), 0, "")


def header_struct_size(name):
    """sizeof of a header struct computed from its field list (LP64: int64_t 8, int32_t 4, pointers 8)."""
    text = open(os.path.join(ROOT, "include", "trepb.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    size = 0
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        n = len(decl.split(","))
        if "*" in decl:
            size = (size + 7) // 8 * 8 + 8 * n
        elif decl.startswith("int64_t"):
            size = (size + 7) // 8 * 8 + 8 * n
        else:
            assert decl.startswith("int32_t"), decl
            size += 4 * n
    return (size + 7) // 8 * 8


def test_ctypes_structs_match_the_header():
    assert C.sizeof(L.TangentArgs) == header_struct_size("trepb_tangent_args") == 8 + 4 * 4 + 8 * 8
    assert C.sizeof(L.AdjointArgs) == header_struct_size("trepb_adjoint_args") == 8 + 4 * 4 + 8 * 8
    assert [f for f, _ in L.TangentArgs._fields_] == ["batch", "nsteps", "nX", "nU", "_pad", "A", "B", "K", "bdX",
                                                      "bdU", "x0", "dX", "dU"]
    assert [f for f, _ in L.AdjointArgs._fields_] == ["batch", "nsteps", "nX", "nU", "_pad", "A", "B", "K", "l_dx",
                                                      "l_du", "m_dx", "z", "z1"]
