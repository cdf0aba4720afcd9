"""Per-instance physical parameters on the cooperative kernels, without a GPU: the link-level condensation
(trep_b200/csrc/trepb_coop_sys.h) split into a plan and a numeric evaluation, against coop_pack of the description
rebuilt with each row's numbers, and the blobs of the golden systems against CRCs taken before the split."""
import ctypes as C
import os
import re
import subprocess
import zlib

import numpy as np
import pytest

import golden_util as G
from test_varied_params import variable_refs
from trep_b200 import desc as D
from trep_b200 import lib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(HERE, "_build", "libcoopvariedcheck.so")
SRC = os.path.join(HERE, "coop_varied_check.cc")
DEPS = [SRC, os.path.join(ROOT, "include", "trepb.h")] + [
    os.path.join(ROOT, "trep_b200", "csrc", f)
    for f in ("trepb_coop_sys.h", "trepb_varied.h", "trepb_codegen.h", "trepb_pack.h", "trepb_sys.h")]

# zlib.crc32 of coop_pack's blob followed by grav[3], as the condensation computed it before the plan / evaluation split
BLOB_CRC = {
    "damped_pendulum": (1064, 0xc6b4c62f), "damper_only": (1256, 0xb17f7d33), "dual_pendulums": (1256, 0xa776d8fd),
    "fourbar": (1592, 0xefc52d31), "loop3d": (2536, 0x8ff980b9), "pccd": (2904, 0xe1e40f59),
    "pend_on_cart1": (1224, 0xbed251f4), "pend_on_cart2": (1240, 0xf950311d), "pendulum1": (1064, 0x40f136c8),
    "pendulum5": (2184, 0x92c57ccb), "puppet": (12616, 0x483f6790), "rod": (1720, 0xf29c0a09),
    "spline_pendulum": (1560, 0x7271e1ab), "spring_arms": (2872, 0xdf1f2cde), "tase_pendulum": (1064, 0x36503744),
    "wrench_arm": (2136, 0x056bf4d3),
}
CAP = 1 << 20


def _harness():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if not os.path.exists(SO) or any(os.path.getmtime(x) > os.path.getmtime(SO) for x in DEPS):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-o", SO])
    h = C.CDLL(SO)
    h.cvc_blob.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    h.cvc_expand.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    return h


def _blob(h, d):
    cd, keep = D.to_c(d)
    out = np.zeros(CAP, np.uint8)
    n = h.cvc_blob(C.byref(cd), out.ctypes.data, CAP)
    return out[:n].tobytes() if n > 0 else None


@pytest.mark.parametrize("name", sorted(BLOB_CRC))
def test_blob_unchanged(name):
    blob = _blob(_harness(), G.desc(name))
    assert (len(blob), zlib.crc32(blob)) == BLOB_CRC[name]


def _rotation_angles(d):
    return [(D.PAR_TABLES["frame_value"], f) for f in range(len(d.frame_kind))
            if d.frame_config[f] < 0 and D.RX <= d.frame_kind[f] <= D.RZ and d.frame_value[f] != 0.0]


@pytest.mark.parametrize("name", sorted(BLOB_CRC))
def test_evaluation_equals_coop_pack_of_the_rebuilt_description(name):
    """Random rows over every variable entry (rotation angles included: both sides use the C library's cos / sin
    here): the plan evaluated on the expansion of the row equals coop_pack of the description with the row's
    numbers, byte for byte; a row of no entries gives the description's own blob."""
    h = _harness()
    d = G.desc(name)
    cd, keep = D.to_c(d)
    out = np.zeros(CAP, np.uint8)
    n = h.cvc_expand(C.byref(cd), 0, None, None, None, out.ctypes.data, CAP)
    assert out[:n].tobytes() == _blob(h, d)
    rng = np.random.default_rng(zlib.crc32(name.encode()) + 1)
    allv = variable_refs(d)
    for draw in range(8):
        refs = allv if draw == 0 else [allv[i] for i in rng.choice(len(allv), int(rng.integers(1, len(allv) + 1)), replace=False)]
        refs = list(dict.fromkeys(refs + _rotation_angles(d)))
        t = np.array([r[0] for r in refs], np.int32)
        i = np.array([r[1] for r in refs], np.int32)
        row = np.array([d.param_value(r) for r in refs]) * rng.uniform(0.5, 1.5, len(refs))
        n = h.cvc_expand(C.byref(cd), len(refs), t.ctypes.data, i.ctypes.data, row.ctypes.data, out.ctypes.data, CAP)
        want = _blob(h, d.with_params(refs, row))
        assert n > 0 and out[:n].tobytes() == want, (name, draw)


def test_flag_mirrors_the_header():
    text = open(os.path.join(ROOT, "include", "trepb.h")).read()
    v = int(re.search(r"#define TREPB_FLAG_COOP_VARIED (\d+)", text).group(1))
    assert v == 128 == lib.FLAG_COOP_VARIED
    flags = [int(x) for x in re.findall(r"#define TREPB_FLAG_\w+ (\d+)", text)]
    assert len(flags) == len(set(flags))
