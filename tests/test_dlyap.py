"""Argument validation of the closed-loop Lyapunov solve (trepb_dlyap_batch[_dev]) and the layout of its argument
struct.  Every refusal happens before any CUDA call, so these run without a device: the exact return code and
trepb_last_error() text of each refused input, and TREPB_OK for an empty batch.  The shape limit (nX above what
shared memory holds) needs the device's opt-in limit and is checked in test_gpu_dlyap.py."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from trep_b200 import lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INVALID = 1
FAKE = 0x1000          # a non-null address: never dereferenced by a refused call or an empty batch
ARRAYS = ("A", "B", "K", "Q", "R", "S", "gain_index", "model_index", "x0", "W", "P", "cost", "status", "iterations")
REQUIRED = ("A", "B", "K", "Q", "R", "status")
IDS = ["host", "dev"]


def dlyap_args(pairs=3, gains=3, models=3, nX=4, nU=1, max_iterations=64, tol=1e-13, null=("W",)):
    a = L.DlyapArgs(pairs=pairs, gains=gains, models=models, nX=nX, nU=nU, max_iterations=max_iterations, tol=tol)
    for f in ARRAYS:
        setattr(a, f, None if f in null else FAKE)
    return a


def call(dev, a):
    ptr = None if a is None else C.byref(a)
    return L.raw().trepb_dlyap_batch_dev(0, ptr, None) if dev else L.raw().trepb_dlyap_batch(0, ptr)


def expect(rc, code, msg):
    assert rc == code
    if code:
        assert L.raw().trepb_last_error().decode() == msg


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
def test_null_argument_is_refused(dev):
    expect(call(dev, None), INVALID, "null argument")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
@pytest.mark.parametrize("sizes", [dict(pairs=-1), dict(gains=-1), dict(models=-1), dict(nX=0), dict(nX=-2),
                                   dict(nU=0), dict(max_iterations=0), dict(max_iterations=-1)],
                         ids=["pairs", "gains", "models", "nX=0", "nX<0", "nU", "max_iterations=0",
                              "max_iterations<0"])
def test_bad_sizes_are_refused(dev, sizes):
    expect(call(dev, dlyap_args(**sizes)), INVALID, "bad sizes")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
@pytest.mark.parametrize("tol", [0.0, -1e-13, float("nan"), float("-inf")], ids=["zero", "negative", "nan", "-inf"])
def test_a_non_positive_tolerance_is_refused(dev, tol):
    expect(call(dev, dlyap_args(tol=tol)), INVALID, "tol must be positive")
    expect(call(dev, dlyap_args(pairs=0, tol=tol)), INVALID, "tol must be positive")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
def test_each_missing_array_is_named(dev):
    msg = "A, B, K, Q, R and status are required (missing: %s)"
    for f in REQUIRED:
        expect(call(dev, dlyap_args(null=(f, "W"))), INVALID, msg % f)
    expect(call(dev, dlyap_args(null=("B", "K", "status", "W"))), INVALID, msg % "B, K, status")
    expect(call(dev, dlyap_args(pairs=0, null=REQUIRED + ("W",))), INVALID, msg % "A, B, K, Q, R, status")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
def test_the_cost_weights(dev):
    expect(call(dev, dlyap_args(null=())), INVALID, "x0 and W are exclusive")
    expect(call(dev, dlyap_args(null=("x0", "W"))), INVALID, "cost needs x0 or W")
    # without cost neither is needed
    expect(call(dev, dlyap_args(pairs=0, null=("cost", "x0", "W"))), 0, "")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
def test_the_order_of_the_checks(dev):
    # sizes before the tolerance before the arrays before the cost weights before the pair counts
    expect(call(dev, dlyap_args(nX=0, tol=0.0, null=("A",))), INVALID, "bad sizes")
    expect(call(dev, dlyap_args(tol=0.0, null=("A",))), INVALID, "tol must be positive")
    expect(call(dev, dlyap_args(gains=0, null=("A", "x0", "W"))), INVALID,
           "A, B, K, Q, R and status are required (missing: A)")
    expect(call(dev, dlyap_args(gains=0, null=("x0", "W", "gain_index"))), INVALID, "cost needs x0 or W")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
def test_without_an_index_every_pair_needs_its_own_gain_and_model(dev):
    expect(call(dev, dlyap_args(pairs=4, gains=3, null=("W", "gain_index"))), INVALID,
           "without gain_index pair p evaluates gain p: gains must be >= pairs")
    expect(call(dev, dlyap_args(pairs=4, gains=4, models=3, null=("W", "model_index"))), INVALID,
           "without model_index pair p runs under model p: models must be >= pairs")


@pytest.mark.parametrize("which", ["gain_index", "model_index"])
@pytest.mark.parametrize("bad", [-1, 5, 2 ** 31 - 1], ids=["negative", "count", "int_max"])
def test_an_index_out_of_range_is_refused_by_the_host_entry(which, bad):
    """The host entry reads the indices before any CUDA call; the _dev entry cannot, and its kernel reports the pair
    as DLYAP_BAD_INDEX instead (test_gpu_dlyap.py)."""
    idx = np.zeros(7, np.int32)
    idx[3] = bad
    ok = np.zeros(7, np.int32)
    a = dlyap_args(pairs=7, gains=5, models=5)
    a.gain_index = (idx if which == "gain_index" else ok).ctypes.data
    a.model_index = (idx if which == "model_index" else ok).ctypes.data
    expect(call(False, a), INVALID, "%s[3] = %d is outside [0, 5)" % (which, bad))


def test_an_index_into_no_gains_is_refused():
    idx = np.zeros(2, np.int32)
    a = dlyap_args(pairs=2, gains=0, models=2, null=("W", "model_index"))
    a.gain_index = idx.ctypes.data
    expect(call(False, a), INVALID, "gain_index[0] = 0 is outside [0, 0)")


@pytest.mark.parametrize("dev", [False, True], ids=IDS)
def test_empty_batch_succeeds(dev):
    expect(call(dev, dlyap_args(pairs=0, gains=0, models=0)), 0, "")
    # the optional arrays may be null
    opt = ("S", "gain_index", "model_index", "x0", "W", "P", "cost", "iterations")
    expect(call(dev, dlyap_args(pairs=0, null=opt)), 0, "")


def header_struct(name):
    """(sizeof, [(field, offset)]) of a header struct from its field list (LP64: int64_t, double and pointers 8
    bytes and 8-aligned, int32_t 4)."""
    text = open(os.path.join(ROOT, "include", "trepb.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    size, fields = 0, []
    for decl in filter(None, (d.strip() for d in body.split(";"))):
        names = [n.strip().lstrip("*").strip() for n in re.sub(r"^(const\s+)?\w+\s*\*?", "", decl).split(",")]
        wide = "*" in decl or decl.startswith(("int64_t", "double"))
        assert wide or decl.startswith("int32_t"), decl
        if wide:
            size = (size + 7) // 8 * 8
        for n in names:
            fields.append((n, size))
            size += 8 if wide else 4
    return (size + 7) // 8 * 8, fields


def test_ctypes_struct_matches_the_header():
    size, fields = header_struct("trepb_dlyap_args")
    assert C.sizeof(L.DlyapArgs) == size == 3 * 8 + 7 * 4 + 4 + 8 + 14 * 8
    assert [f for f, _ in L.DlyapArgs._fields_] == [f for f, _ in fields]
    assert [(f, getattr(L.DlyapArgs, f).offset) for f, _ in L.DlyapArgs._fields_] == fields
    assert [f for f, _ in fields] == ["pairs", "gains", "models", "nX", "nU", "max_iterations", "q_per_model",
                                      "r_per_model", "s_per_model", "x0_per_pair", "tol"] + list(ARRAYS)


def test_status_codes_match_the_header():
    text = open(os.path.join(ROOT, "include", "trepb.h")).read()
    code = lambda n: int(re.search(r"#define TREPB_DLYAP_%s (-?\d+)" % n, text).group(1))
    assert (L.DLYAP_STABLE, L.DLYAP_NOT_CONVERGED, L.DLYAP_NONFINITE, L.DLYAP_BAD_INDEX) == \
        (code("STABLE"), code("NOT_CONVERGED"), code("NONFINITE"), code("BAD_INDEX")) == (0, -1, -3, -4)
    assert set(L.DLYAP_STATUS) == {0, -1, -3, -4}


def test_the_new_entry_points_are_exported():
    for n in ("trepb_dlyap_batch", "trepb_dlyap_batch_dev"):
        assert n in L.EXPORTS and hasattr(L.raw(), n)


def test_solve_closed_loop_needs_the_pairs_spelled_out():
    with pytest.raises(ValueError, match="3 gains and 2 models"):
        L.solve_closed_loop(np.zeros((2, 4, 4)), np.zeros((2, 4, 1)), np.zeros((3, 1, 4)), np.eye(4), np.eye(1))
    with pytest.raises(ValueError, match="gain_index has 2 pairs, model_index 3"):
        L.solve_closed_loop(np.zeros((2, 4, 4)), np.zeros((2, 4, 1)), np.zeros((3, 1, 4)), np.eye(4), np.eye(1),
                            gain_index=[0, 1], model_index=[0, 1, 1])
