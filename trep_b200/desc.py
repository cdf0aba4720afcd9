"""Flat, Python-object-free description of a mechanical system.

This is the host-side "synchronize" product: what the reference computes in
``trep/system.py:672-840`` (frame order = pre-order DFS, ``configs = dyn + kin``,
``config_gen``, ``masses``) and ``trep/frame.py:658-721`` (``cache_index``), reduced to the
plain arrays the C ABI (`include/trepb.h`, ``trepb_sysdesc``) takes.  Nothing in here
touches a GPU; it is the input of ``trepb_system_create``.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import json
from dataclasses import dataclass, field

import numpy as np

# frame kinds (trep/_trep/trep.h:168-273 transform types)
WORLD, TX, TY, TZ, RX, RY, RZ, CONST_SE3 = range(8)
KIND_NAMES = ["WORLD", "TX", "TY", "TZ", "RX", "RY", "RZ", "CONST_SE3"]

# potential kinds
POT_GRAVITY, POT_LINEAR_SPRING, POT_CONFIG_SPRING, POT_NONLINEAR_CONFIG_SPRING = range(4)
# force kinds
FORCE_DAMPING, FORCE_CONFIG, FORCE_LINEAR_DAMPER, FORCE_BODY_WRENCH, FORCE_HYBRID_WRENCH, FORCE_SPATIAL_WRENCH = range(6)
# constraint kinds
CON_DISTANCE, CON_POINT1D, CON_PLANE = range(3)
# tables a per-instance parameter can come from (TREPB_PAR_*, include/trepb.h)
PAR_TABLE_NAMES = ["frame_value", "frame_se3", "frame_mass", "pot_d", "force_d", "con_d", "dpool"]
PAR_TABLES = {n: i for i, n in enumerate(PAR_TABLE_NAMES)}


@dataclass
class SystemDesc:
    """All arrays are C-contiguous; frame 0 is the world frame."""
    frame_parent: np.ndarray          # int32 [nF]   (-1 for world)
    frame_kind: np.ndarray            # int32 [nF]
    frame_config: np.ndarray          # int32 [nF]   (-1: constant transform)
    frame_value: np.ndarray           # f64   [nF]   constant parameter of a primitive transform
    frame_se3: np.ndarray             # f64   [nF,12] row-major 3x4 [R|p]; identity unless CONST_SE3
    frame_mass: np.ndarray            # f64   [nF,4]  m, Ixx, Iyy, Izz
    nd: int
    nk: int
    nu: int
    pot_kind: np.ndarray              # int32 [nP]
    pot_i: np.ndarray                 # int32 [nP,4]
    pot_d: np.ndarray                 # f64   [nP,4]
    force_kind: np.ndarray            # int32 [nFo]
    force_i: np.ndarray               # int32 [nFo,4]
    force_d: np.ndarray               # f64   [nFo,4]
    con_kind: np.ndarray              # int32 [nc]
    con_i: np.ndarray                 # int32 [nc,4]
    con_d: np.ndarray                 # f64   [nc,4]   [distance | n0, tolerance, n1, n2]
    ipool: np.ndarray                 # int32 [*]  variable-length int payloads (tape-measure paths)
    dpool: np.ndarray                 # f64   [*]  variable-length double payloads (damping coefficients)
    frame_names: list = field(default_factory=list)
    config_names: list = field(default_factory=list)
    input_names: list = field(default_factory=list)
    name: str = ""

    # ---- sizes ---------------------------------------------------------------------------
    @property
    def n_frames(self):
        return int(self.frame_parent.shape[0])

    @property
    def nq(self):
        return self.nd + self.nk

    @property
    def nc(self):
        return int(self.con_kind.shape[0])

    @property
    def nX(self):
        """DSystem state size  [Q(nq); p(nd); v(nk)]  (trep/discopt/dsystem.py:40-66)."""
        return 2 * self.nq

    @property
    def nU(self):
        """DSystem input size  [u(nu); rho(nk)]."""
        return self.nu + self.nk

    # ---- derived structure (what frame.py:683-691 calls cache_index) ----------------------
    def ancestors(self, f):
        """Config indices driving frame ``f``'s position, ordered root -> leaf."""
        out = []
        while f >= 0:
            c = int(self.frame_config[f])
            if c >= 0:
                out.append(c)
            f = int(self.frame_parent[f])
        return out[::-1]

    def config_frame(self):
        """frame index driven by each config (-1 for non-frame configs, e.g. string lengths)."""
        cf = -np.ones(self.nq, dtype=np.int32)
        for f in range(self.n_frames):
            c = int(self.frame_config[f])
            if c >= 0:
                cf[c] = f
        return cf

    def mass_frames(self):
        m = self.frame_mass
        return [f for f in range(self.n_frames) if np.any(m[f] != 0.0)]

    # ---- (de)serialisation ---------------------------------------------------------------
    _ARRAYS = ["frame_parent", "frame_kind", "frame_config", "frame_value", "frame_se3",
               "frame_mass", "pot_kind", "pot_i", "pot_d", "force_kind", "force_i", "force_d",
               "con_kind", "con_i", "con_d", "ipool", "dpool"]

    def to_json(self):
        d = {k: getattr(self, k).tolist() for k in self._ARRAYS}
        # doubles are written with repr() by json -> exact round trip
        d.update(nd=self.nd, nk=self.nk, nu=self.nu, frame_names=self.frame_names,
                 config_names=self.config_names, input_names=self.input_names, name=self.name)
        return json.dumps(d)

    @staticmethod
    def from_json(text):
        d = json.loads(text)
        return make_desc(**d)

    def save(self, path):
        with open(path, "w") as fh:
            fh.write(self.to_json())

    @staticmethod
    def load(path):
        with open(path) as fh:
            return SystemDesc.from_json(fh.read())

    def structural_hash(self):
        """Hash over everything that changes generated code (topology AND parameters)."""
        h = hashlib.sha256()
        for k in self._ARRAYS:
            a = getattr(self, k)
            h.update(k.encode())
            h.update(str(a.shape).encode())
            h.update(np.ascontiguousarray(a).tobytes())
        h.update(("%d,%d,%d" % (self.nd, self.nk, self.nu)).encode())
        return h.hexdigest()[:16]

    # ---- per-instance parameters (trepb_varied, include/trepb.h) ---------------------------
    def param_ref(self, table, *idx):
        """(TREPB_PAR_* id, flat index) of one numeric entry, for per-instance parameters.  table: a key of
        PAR_TABLES; idx: the entry's index in that array - a frame name or index (+ component) for the frame
        tables, e.g. param_ref("frame_mass", "Pendulum", 0) or param_ref("pot_d", 0, 2)."""
        if table not in PAR_TABLES:
            raise ValueError("unknown parameter table %r (one of %s)" % (table, ", ".join(PAR_TABLES)))
        idx = list(idx)
        if table.startswith("frame_") and idx and isinstance(idx[0], str):
            if idx[0] not in self.frame_names:
                raise ValueError("no frame named %r" % idx[0])
            idx[0] = self.frame_names.index(idx[0])
        a = getattr(self, table)
        if len(idx) != a.ndim:
            raise ValueError("%s takes %d index(es)" % (table, a.ndim))
        return PAR_TABLES[table], int(np.ravel_multi_index(tuple(int(i) for i in idx), a.shape))

    def param_value(self, ref):
        """The description's value of a param_ref."""
        t, i = ref
        return float(getattr(self, PAR_TABLE_NAMES[t]).reshape(-1)[i])

    def with_params(self, refs, values):
        """A copy with the entries `refs` set to `values` (one row of a per-instance parameter array)."""
        arrs = {k: getattr(self, k).copy() for k in self._ARRAYS}
        for (t, i), v in zip(refs, values):
            arrs[PAR_TABLE_NAMES[t]].reshape(-1)[i] = v
        return SystemDesc(**arrs, nd=self.nd, nk=self.nk, nu=self.nu, frame_names=list(self.frame_names),
                          config_names=list(self.config_names), input_names=list(self.input_names), name=self.name)

    def equal(self, other):
        if (self.nd, self.nk, self.nu) != (other.nd, other.nk, other.nu):
            return False
        for k in self._ARRAYS:
            a, b = getattr(self, k), getattr(other, k)
            if a.shape != b.shape or not np.array_equal(a, b):
                return False
        return True


def _arr(x, dtype, shape_tail=None):
    a = np.ascontiguousarray(np.array(x, dtype=dtype))
    if shape_tail is not None:
        a = a.reshape((-1,) + tuple(shape_tail))
    return a


def make_desc(frame_parent, frame_kind, frame_config, frame_value, frame_se3, frame_mass,
              nd, nk, nu, pot_kind=(), pot_i=(), pot_d=(), force_kind=(), force_i=(),
              force_d=(), con_kind=(), con_i=(), con_d=(), ipool=(), dpool=(),
              frame_names=None, config_names=None, input_names=None, name=""):
    d = SystemDesc(
        frame_parent=_arr(frame_parent, np.int32), frame_kind=_arr(frame_kind, np.int32),
        frame_config=_arr(frame_config, np.int32), frame_value=_arr(frame_value, np.float64),
        frame_se3=_arr(frame_se3, np.float64, (12,)), frame_mass=_arr(frame_mass, np.float64, (4,)),
        nd=int(nd), nk=int(nk), nu=int(nu),
        pot_kind=_arr(pot_kind, np.int32), pot_i=_arr(pot_i, np.int32, (4,)),
        pot_d=_arr(pot_d, np.float64, (4,)),
        force_kind=_arr(force_kind, np.int32), force_i=_arr(force_i, np.int32, (4,)),
        force_d=_arr(force_d, np.float64, (4,)),
        con_kind=_arr(con_kind, np.int32), con_i=_arr(con_i, np.int32, (4,)),
        con_d=_arr(con_d, np.float64, (4,)),
        ipool=_arr(ipool, np.int32), dpool=_arr(dpool, np.float64),
        frame_names=list(frame_names or []), config_names=list(config_names or []),
        input_names=list(input_names or []), name=name)
    validate(d)
    return d


def validate(d: SystemDesc):
    nF = d.n_frames
    if nF < 1 or d.frame_kind[0] != WORLD or d.frame_parent[0] != -1:
        raise ValueError("frame 0 must be the world frame")
    for f in range(1, nF):
        p = int(d.frame_parent[f])
        if not (0 <= p < f):
            raise ValueError("frames must be in pre-order (parent before child): frame %d" % f)
        k = int(d.frame_kind[f])
        if not (TX <= k <= CONST_SE3):
            raise ValueError("frame %d: unknown transform kind %d" % (f, k))
        c = int(d.frame_config[f])
        if c >= d.nq or c < -1:
            raise ValueError("frame %d: config index out of range" % f)
        if k == CONST_SE3 and c >= 0:
            raise ValueError("CONST_SE3 frames cannot be driven by a config")
    cfgs = [int(c) for c in d.frame_config if c >= 0]
    if len(set(cfgs)) != len(cfgs):
        raise ValueError("a config may drive only one frame")
    for a, n in ((d.pot_i, len(d.pot_kind)), (d.force_i, len(d.force_kind)), (d.con_i, len(d.con_kind))):
        if a.shape[0] != n:
            raise ValueError("record arrays disagree in length")


# ------------------------------------------------------------------------------------------
# ctypes mirror of `trepb_sysdesc` (include/trepb.h)
# ------------------------------------------------------------------------------------------
class CSysDesc(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int32), ("nd", C.c_int32), ("nk", C.c_int32), ("nu", C.c_int32),
        ("n_potentials", C.c_int32), ("n_forces", C.c_int32), ("n_constraints", C.c_int32),
        ("n_ipool", C.c_int32), ("n_dpool", C.c_int32), ("_pad", C.c_int32),
        ("frame_parent", C.POINTER(C.c_int32)), ("frame_kind", C.POINTER(C.c_int32)),
        ("frame_config", C.POINTER(C.c_int32)), ("frame_value", C.POINTER(C.c_double)),
        ("frame_se3", C.POINTER(C.c_double)), ("frame_mass", C.POINTER(C.c_double)),
        ("pot_kind", C.POINTER(C.c_int32)), ("pot_i", C.POINTER(C.c_int32)),
        ("pot_d", C.POINTER(C.c_double)),
        ("force_kind", C.POINTER(C.c_int32)), ("force_i", C.POINTER(C.c_int32)),
        ("force_d", C.POINTER(C.c_double)),
        ("con_kind", C.POINTER(C.c_int32)), ("con_i", C.POINTER(C.c_int32)),
        ("con_d", C.POINTER(C.c_double)),
        ("ipool", C.POINTER(C.c_int32)), ("dpool", C.POINTER(C.c_double)),
    ]


def to_c(d: SystemDesc):
    """Returns (CSysDesc, keepalive) — keep `keepalive` referenced while the struct is in use."""
    keep = []

    def ip(a):
        a = np.ascontiguousarray(a, dtype=np.int32)
        keep.append(a)
        return a.ctypes.data_as(C.POINTER(C.c_int32))

    def dp(a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        keep.append(a)
        return a.ctypes.data_as(C.POINTER(C.c_double))

    s = CSysDesc(
        n_frames=d.n_frames, nd=d.nd, nk=d.nk, nu=d.nu,
        n_potentials=len(d.pot_kind), n_forces=len(d.force_kind), n_constraints=len(d.con_kind),
        n_ipool=len(d.ipool), n_dpool=len(d.dpool), _pad=0,
        frame_parent=ip(d.frame_parent), frame_kind=ip(d.frame_kind), frame_config=ip(d.frame_config),
        frame_value=dp(d.frame_value), frame_se3=dp(d.frame_se3), frame_mass=dp(d.frame_mass),
        pot_kind=ip(d.pot_kind), pot_i=ip(d.pot_i), pot_d=dp(d.pot_d),
        force_kind=ip(d.force_kind), force_i=ip(d.force_i), force_d=dp(d.force_d),
        con_kind=ip(d.con_kind), con_i=ip(d.con_i), con_d=dp(d.con_d),
        ipool=ip(d.ipool), dpool=dp(d.dpool))
    return s, keep
