"""Per-instance physical parameters (trepb_*_varied_batch*) without a GPU: which entries may vary, the ctypes
mirror of trepb_varied, and the expansion the kernels read (trep_b200/csrc/trepb_varied.h) against re-packing the
description rebuilt with each instance's numbers."""
import ctypes as C
import os
import re
import subprocess
import zlib

import numpy as np
import pytest

import golden_util as G
from trep_b200 import desc as D
from trep_b200 import lib

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(HERE, "_build", "libvariedcheck.so")
SRC = os.path.join(HERE, "varied_check.cc")
DEPS = [SRC, os.path.join(ROOT, "include", "trepb.h")] + [
    os.path.join(ROOT, "trep_b200", "csrc", f) for f in ("trepb_varied.h", "trepb_codegen.h", "trepb_pack.h", "trepb_sys.h")]

SYSTEMS = G.ALL + G.EXTRA + G.PARITY + G.PARITY_SPRING


def variable_refs(d):
    """Every entry the semantics let vary: non-zero, not +-1 in frame_se3, not a spline x-point."""
    xpts = set()
    for p, k in enumerate(d.pot_kind):
        if k == D.POT_NONLINEAR_CONFIG_SPRING:
            xpts.update(range(int(d.pot_i[p, 1]), int(d.pot_i[p, 1]) + int(d.pot_i[p, 2])))
    refs = []
    for t, name in enumerate(D.PAR_TABLE_NAMES):
        for i, v in enumerate(getattr(d, name).reshape(-1)):
            if v == 0.0 or (name == "frame_se3" and abs(v) == 1.0) or (name == "dpool" and i in xpts):
                continue
            refs.append((t, i))
    return refs


def test_check_params_accepts_every_run_time_entry():
    for name in SYSTEMS:
        d = G.desc(name)
        refs = variable_refs(d)
        assert refs, name
        lib.check_params(d, refs)
        for r in refs:
            assert d.param_value(r) != 0.0


def _refused(d, refs, pattern):
    with pytest.raises(lib.TrepbError) as e:
        lib.check_params(d, refs)
    assert e.value.code == 1
    assert re.search(pattern, str(e.value)), str(e.value)


def test_check_params_refuses_structural_entries_by_name():
    d = G.desc("damped_pendulum")
    # frame 3 carries m = 1 and no rotational inertia: Ixx is a literal zero
    _refused(d, [d.param_ref("pot_d", 0, 2), d.param_ref("frame_mass", 3, 1)], r"entry 1 \(FRAME_MASS\[13\]\).*value is 0")
    _refused(d, [d.param_ref("dpool", 0), d.param_ref("dpool", 0)], r"entry 1 \(DPOOL\[0\]\).*more than once")
    _refused(d, [(D.PAR_TABLES["frame_mass"], 16)], r"FRAME_MASS\[16\].*out of range")
    _refused(d, [(D.PAR_TABLES["dpool"], -1)], r"DPOOL\[-1\].*out of range")
    _refused(d, [(7, 0)], r"unknown table")
    w = G.desc("wrench_arm")
    f = int(np.flatnonzero(w.frame_kind == D.CONST_SE3)[0])
    k = int(np.flatnonzero(np.abs(w.frame_se3[f]) == 1.0)[0])
    _refused(w, [w.param_ref("frame_se3", f, k)], r"FRAME_SE3\[%d\].*\+-1" % (12 * f + k))
    s = G.desc("spline_pendulum")
    p = int(np.flatnonzero(s.pot_kind == D.POT_NONLINEAR_CONFIG_SPRING)[0])
    x0 = int(s.pot_i[p, 1])
    _refused(s, [s.param_ref("dpool", x0 + 1)], r"DPOOL\[%d\].*spline x-point" % (x0 + 1))
    c0 = x0 + int(s.pot_i[p, 2])
    c = c0 + int(np.flatnonzero(s.dpool[c0:] != 0.0)[0])
    lib.check_params(s, [s.param_ref("dpool", c)])   # spline coefficients may vary


def test_param_ref_takes_frame_names():
    d = G.desc("puppet")
    f = next(i for i, n in enumerate(d.frame_names) if n and np.any(d.frame_mass[i] != 0))
    assert d.param_ref("frame_mass", d.frame_names[f], 0) == (D.PAR_TABLES["frame_mass"], 4 * f)
    assert d.param_value(d.param_ref("frame_mass", d.frame_names[f], 0)) == d.frame_mass[f, 0]
    with pytest.raises(ValueError):
        d.param_ref("frame_mass", "no such frame", 0)


def test_varied_mirror_matches_the_header():
    text = open(os.path.join(ROOT, "include", "trepb.h")).read()
    body = re.search(r"typedef struct trepb_varied \{(.*?)\} trepb_varied;", text, re.S).group(1)
    decl = re.findall(r"^\s*(?:const\s+)?(int32_t|double)\s*(\*?)\s*([\w, ]+);", body, re.M)
    names = [n.strip() for _, _, ns in decl for n in ns.split(",")]
    assert names == [f[0] for f in lib.Varied._fields_]
    assert C.sizeof(lib.Varied) == 32
    assert [getattr(lib.Varied, n).offset for n in names] == [0, 4, 8, 16, 24]
    ids = dict(re.findall(r"#define TREPB_PAR_(\w+)\s+(\d+)", text))
    assert {n.upper(): str(i) for n, i in D.PAR_TABLES.items()} == ids


def _harness():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    if not os.path.exists(SO) or any(os.path.getmtime(x) > os.path.getmtime(SO) for x in DEPS):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", SRC, "-o", SO])
    h = C.CDLL(SO)
    h.vc_expand.restype = C.c_int
    h.vc_packed.restype = C.c_int
    return h


@pytest.mark.parametrize("name", SYSTEMS)
def test_expansion_equals_repacking(name):
    """For random draws (+-50 % around the base, a Gravity component and a Damping coefficient always among them where
    the system has one), the expansion of (base description, entries, row) equals, byte for byte, param_map(pack(
    desc_b)).values and the numeric region of pack(desc_b).blob + grav, desc_b = the description with the row's
    numbers."""
    h = _harness()
    d = G.desc(name)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    allv = variable_refs(d)
    must = [r for r in allv if r[0] == D.PAR_TABLES["pot_d"] and d.pot_kind[r[1] // 4] == D.POT_GRAVITY]
    damp = [int(d.force_i[f, 0]) for f in range(len(d.force_kind)) if d.force_kind[f] == D.FORCE_DAMPING]
    must += [r for r in allv if r[0] == D.PAR_TABLES["dpool"] and damp and damp[0] <= r[1] < damp[0] + d.nd][:1]
    cd, keep = D.to_c(d)
    for draw in range(6):
        k = int(rng.integers(1, len(allv) + 1))
        pick = [allv[i] for i in rng.choice(len(allv), size=k, replace=False)]
        refs = list(dict.fromkeys(must[:1 + draw % 2] + pick))
        t = np.array([r[0] for r in refs], np.int32)
        i = np.array([r[1] for r in refs], np.int32)
        row = np.array([d.param_value(r) for r in refs]) * rng.uniform(0.5, 1.5, len(refs))
        db = d.with_params(refs, row)
        cdb, keepb = D.to_c(db)
        for slots in (1, 0):
            out = np.zeros(20000)
            n = h.vc_expand(C.byref(cd), len(refs), t.ctypes.data, i.ctypes.data, slots, row.ctypes.data,
                            out.ctypes.data, out.size)
            want = np.zeros(20000)
            m = h.vc_packed(C.byref(cdb), slots, want.ctypes.data, want.size)
            assert n == m > 0, (name, slots, n, m)
            assert out[:n].tobytes() == want[:m].tobytes(), (name, draw, slots)


def test_no_variation_expands_to_the_base():
    h = _harness()
    for name in SYSTEMS:
        d = G.desc(name)
        cd, keep = D.to_c(d)
        for slots in (1, 0):
            out, want = np.zeros(20000), np.zeros(20000)
            n = h.vc_expand(C.byref(cd), 0, None, None, slots, None, out.ctypes.data, out.size)
            assert n == h.vc_packed(C.byref(cd), slots, want.ctypes.data, want.size)
            assert out[:n].tobytes() == want[:n].tobytes()
