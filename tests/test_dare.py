"""Argument validation of the stationary-LQR solve (trepb_dare_batch[_dev]) and the layout of its argument struct.
Every refusal happens before any CUDA call, so these run without a device: the exact return code and
trepb_last_error() text of each refused input, and TREPB_OK for an empty batch."""
import ctypes as C
import os
import re

import pytest

from trep_b200 import lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID = 1
FAKE = 0x1000          # a non-null address: never dereferenced by a refused call or an empty batch
ARRAYS = ("A", "B", "Q", "R", "S", "K", "P", "status", "iterations")
REQUIRED = ("A", "B", "Q", "R", "status")
IDS = ["host", "dev"]


def dare_args(batch=3, nX=4, nU=1, max_iterations=64, tol=1e-13, **null):
    a = L.DareArgs(batch=batch, nX=nX, nU=nU, max_iterations=max_iterations, tol=tol)
    for f in ARRAYS:
        setattr(a, f, None if f in null else FAKE)
    return a


def call(dev, a):
    ptr = None if a is None else C.byref(a)
    return L.raw().trepb_dare_batch_dev(0, ptr, None) if dev else L.raw().trepb_dare_batch(0, ptr)


def expect(rc, code, msg):
    assert rc == code
    if code:
        assert L.raw().trepb_last_error().decode() == msg


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
def test_null_argument_is_refused(dev):
    expect(call(dev, None), INVALID, "null argument")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
@pytest.mark.parametrize("sizes", [dict(batch=-1), dict(nX=0), dict(nX=-2), dict(nU=0), dict(max_iterations=0),
                                   dict(max_iterations=-1)],
                         ids=["batch", "nX=0", "nX<0", "nU", "max_iterations=0", "max_iterations<0"])
def test_bad_sizes_are_refused(dev, sizes):
    expect(call(dev, dare_args(**sizes)), INVALID, "bad sizes")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
@pytest.mark.parametrize("tol", [0.0, -1e-13, float("nan"), float("-inf")], ids=["zero", "negative", "nan", "-inf"])
def test_a_non_positive_tolerance_is_refused(dev, tol):
    expect(call(dev, dare_args(tol=tol)), INVALID, "tol must be positive")
    expect(call(dev, dare_args(batch=0, tol=tol)), INVALID, "tol must be positive")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
def test_each_missing_array_is_named(dev):
    for f in REQUIRED:
        expect(call(dev, dare_args(**{f: 1})), INVALID,
               "A, B, Q, R and status are required (missing: %s)" % f)
    expect(call(dev, dare_args(A=1, Q=1, status=1)), INVALID,
           "A, B, Q, R and status are required (missing: A, Q, status)")
    expect(call(dev, dare_args(batch=0, **{f: 1 for f in REQUIRED})), INVALID,
           "A, B, Q, R and status are required (missing: A, B, Q, R, status)")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
def test_the_order_of_the_checks(dev):
    # sizes before the tolerance before the arrays
    expect(call(dev, dare_args(nX=0, tol=0.0, A=1)), INVALID, "bad sizes")
    expect(call(dev, dare_args(tol=0.0, A=1)), INVALID, "tol must be positive")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
def test_empty_batch_succeeds(dev):
    expect(call(dev, dare_args(batch=0)), 0, "")
    # the optional arrays may be null
    expect(call(dev, dare_args(batch=0, S=1, K=1, P=1, iterations=1)), 0, "")


def header_struct_size(name):
    """sizeof of a header struct from its field list (LP64: int64_t, double and pointers 8 bytes, int32_t 4)."""
    text = open(os.path.join(ROOT, "include", "trepb.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    size = 0
    for decl in filter(None, (d.strip() for d in body.split(";"))):
        n = len(decl.split(","))
        if "*" in decl or decl.startswith(("int64_t", "double")):
            size = (size + 7) // 8 * 8 + 8 * n
        else:
            assert decl.startswith("int32_t"), decl
            size += 4 * n
    return (size + 7) // 8 * 8


def test_ctypes_struct_matches_the_header():
    assert C.sizeof(L.DareArgs) == header_struct_size("trepb_dare_args") == 8 + 6 * 4 + 8 + 9 * 8
    assert [f for f, _ in L.DareArgs._fields_] == ["batch", "nX", "nU", "max_iterations", "q_per_rollout",
                                                   "r_per_rollout", "s_per_rollout", "tol"] + list(ARRAYS)


def test_status_codes_match_the_header():
    text = open(os.path.join(ROOT, "include", "trepb.h")).read()
    code = lambda n: int(re.search(r"#define TREPB_DARE_%s (-?\d+)" % n, text).group(1))
    assert (L.DARE_OK, L.DARE_NOT_CONVERGED, L.DARE_SINGULAR, L.DARE_NONFINITE) == \
        (code("OK"), code("NOT_CONVERGED"), code("SINGULAR"), code("NONFINITE")) == (0, -1, -2, -3)


def test_the_new_entry_points_are_exported():
    for n in ("trepb_dare_batch", "trepb_dare_batch_dev"):
        assert n in L.EXPORTS and hasattr(L.raw(), n)
