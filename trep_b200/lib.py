"""ctypes binding of libtrepb.so (the C ABI declared in include/trepb.h).

There is no fallback: if the library has not been built (``python -m trep_b200.build``) the
import of this module raises, and every compute call needs a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import desc as D

HERE = os.path.dirname(os.path.abspath(__file__))
LIBPATH = os.environ.get("TREPB_LIBPATH") or os.path.join(HERE, "libtrepb.so")

if not os.path.exists(LIBPATH):
    raise ImportError("trep_b200/libtrepb.so is missing: build it with `python -m trep_b200.build` "
                      "(there is no CPU fallback)")
_lib = C.CDLL(LIBPATH)

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class StepArgs(C.Structure):
    _fields_ = [("batch", C.c_int64), ("nsteps", C.c_int32), ("max_iterations", C.c_int32),
                ("t0", C.c_double), ("dt", C.c_double), ("tolerance", C.c_double),
                ("q1", C.c_void_p), ("p1", C.c_void_p), ("u1", C.c_void_p), ("k2", C.c_void_p),
                ("q2_guess", C.c_void_p), ("lambda_guess", C.c_void_p),
                ("q2", C.c_void_p), ("p2", C.c_void_p), ("lambda1", C.c_void_p),
                ("iters", C.c_void_p), ("status", C.c_void_p),
                ("sample_every", C.c_int32), ("_pad", C.c_int32),
                ("traj_q", C.c_void_p), ("traj_p", C.c_void_p), ("times", C.c_void_p)]


class ProjectArgs(C.Structure):
    _fields_ = [("batch", C.c_int64), ("nsteps", C.c_int32), ("max_iterations", C.c_int32),
                ("t0", C.c_double), ("dt", C.c_double), ("tolerance", C.c_double),
                ("bX", C.c_void_p), ("bU", C.c_void_p), ("Kfb", C.c_void_p),
                ("k_per_instance", C.c_int32), ("use_hint", C.c_int32),
                ("X", C.c_void_p), ("U", C.c_void_p),
                ("iters", C.c_void_p), ("status", C.c_void_p), ("fail_step", C.c_void_p), ("times", C.c_void_p)]


class LqrArgs(C.Structure):
    _fields_ = [("batch", C.c_int64), ("nsteps", C.c_int32), ("nX", C.c_int32), ("nU", C.c_int32),
                ("q_per_step", C.c_int32), ("r_per_step", C.c_int32), ("_pad", C.c_int32),
                ("A", C.c_void_p), ("B", C.c_void_p), ("Q", C.c_void_p), ("R", C.c_void_p),
                ("Kfb", C.c_void_p), ("P0", C.c_void_p), ("status", C.c_void_p)]


class LqArgs(C.Structure):
    _fields_ = [("batch", C.c_int64), ("nsteps", C.c_int32), ("nX", C.c_int32), ("nU", C.c_int32),
                ("cost_per_rollout", C.c_int32),
                ("A", C.c_void_p), ("B", C.c_void_p), ("Q", C.c_void_p), ("S", C.c_void_p), ("R", C.c_void_p),
                ("q", C.c_void_p), ("r", C.c_void_p), ("Kfb", C.c_void_p), ("C", C.c_void_p), ("P0", C.c_void_p),
                ("b0", C.c_void_p), ("status", C.c_void_p)]


class TangentArgs(C.Structure):
    _fields_ = [("batch", C.c_int64), ("nsteps", C.c_int32), ("nX", C.c_int32), ("nU", C.c_int32), ("_pad", C.c_int32),
                ("A", C.c_void_p), ("B", C.c_void_p), ("K", C.c_void_p), ("bdX", C.c_void_p), ("bdU", C.c_void_p),
                ("x0", C.c_void_p), ("dX", C.c_void_p), ("dU", C.c_void_p)]


class AdjointArgs(C.Structure):
    _fields_ = [("batch", C.c_int64), ("nsteps", C.c_int32), ("nX", C.c_int32), ("nU", C.c_int32), ("_pad", C.c_int32),
                ("A", C.c_void_p), ("B", C.c_void_p), ("K", C.c_void_p), ("l_dx", C.c_void_p), ("l_du", C.c_void_p),
                ("m_dx", C.c_void_p), ("z", C.c_void_p), ("z1", C.c_void_p)]


class TrackArgs(C.Structure):
    _fields_ = [("batch", C.c_int64), ("nsteps", C.c_int32), ("nX", C.c_int32), ("nU", C.c_int32), ("nref", C.c_int32)]\
        + [(n, C.c_void_p) for n in ("X", "U", "Xd", "Ud", "Q", "R", "ref_index", "dX", "dU", "fdxdx", "fdxdu", "fdudu",
                                     "cost", "dcost", "q", "r", "l_dx", "m_dx", "Qm", "Sm", "Rm")]


class CandidatesArgs(C.Structure):
    _fields_ = [("groups", C.c_int64), ("ncand", C.c_int32), ("nsteps", C.c_int32), ("nX", C.c_int32), ("nU", C.c_int32),
                ("nrollouts", C.c_int64)] \
        + [(n, C.c_void_p) for n in ("rows", "lam", "X", "U", "dX", "dU", "Kproj", "bX", "bU", "Kc")]


class DareArgs(C.Structure):
    _fields_ = [("batch", C.c_int64), ("nX", C.c_int32), ("nU", C.c_int32), ("max_iterations", C.c_int32),
                ("q_per_rollout", C.c_int32), ("r_per_rollout", C.c_int32), ("s_per_rollout", C.c_int32),
                ("tol", C.c_double)] \
        + [(n, C.c_void_p) for n in ("A", "B", "Q", "R", "S", "K", "P", "status", "iterations")]


class DlyapArgs(C.Structure):
    _fields_ = [("pairs", C.c_int64), ("gains", C.c_int64), ("models", C.c_int64), ("nX", C.c_int32),
                ("nU", C.c_int32), ("max_iterations", C.c_int32), ("q_per_model", C.c_int32),
                ("r_per_model", C.c_int32), ("s_per_model", C.c_int32), ("x0_per_pair", C.c_int32),
                ("tol", C.c_double)] \
        + [(n, C.c_void_p) for n in ("A", "B", "K", "Q", "R", "S", "gain_index", "model_index", "x0", "W", "P",
                                     "cost", "status", "iterations")]


RAW = ["q2_dq1", "q2_dp1", "q2_du1", "q2_dk2", "p2_dq1", "p2_dp1", "p2_du1", "p2_dk2",
       "l1_dq1", "l1_dp1", "l1_du1", "l1_dk2"]


class LinArgs(C.Structure):
    _fields_ = ([("batch", C.c_int64), ("max_iterations", C.c_int32), ("traj_len", C.c_int32),
                 ("tolerance", C.c_double), ("t1", C.c_void_p), ("t2", C.c_void_p),
                 ("t1_scalar", C.c_double), ("dt_scalar", C.c_double),
                 ("q1", C.c_void_p), ("p1", C.c_void_p), ("u1", C.c_void_p), ("k2", C.c_void_p),
                 ("q2_guess", C.c_void_p), ("lambda_guess", C.c_void_p),
                 ("q2", C.c_void_p), ("p2", C.c_void_p), ("lambda1", C.c_void_p),
                 ("iters", C.c_void_p), ("status", C.c_void_p), ("A", C.c_void_p), ("B", C.c_void_p)]
                + [(n, C.c_void_p) for n in RAW])


D2_KINDS = ["dq1dq1", "dq1dp1", "dq1du1", "dq1dk2", "dp1dp1", "dp1du1", "dp1dk2", "du1du1", "du1dk2", "dk2dk2"]
D2_WHICH = ["q2", "p2", "l1"]


class D2Args(C.Structure):
    _fields_ = [("lin", LinArgs), ("d2", C.c_void_p * 30), ("z", C.c_void_p), ("fdxdx", C.c_void_p),
                ("fdxdu", C.c_void_p), ("fdudu", C.c_void_p)]


class Varied(C.Structure):
    """ctypes mirror of trepb_varied: per-instance values of n description entries."""
    _fields_ = [("n", C.c_int32), ("_pad", C.c_int32), ("table", C.c_void_p), ("index", C.c_void_p),
                ("values", C.c_void_p)]


def _varied(params):
    """(Varied, keepalive) for params = (refs, values): refs a list of SystemDesc.param_ref results, values
    [rows][len(refs)] (numpy for the host entry points, anything with data_ptr() for the _dev ones)."""
    refs, values = params
    refs = [tuple(r) for r in refs]
    t = np.ascontiguousarray([r[0] for r in refs], dtype=np.int32)
    i = np.ascontiguousarray([r[1] for r in refs], dtype=np.int32)
    if isinstance(values, np.ndarray):
        values = np.ascontiguousarray(values, dtype=np.float64)
        if values.ndim != 2 or values.shape[1] != len(refs):
            raise ValueError("params values must be [rows][%d]" % len(refs))
    v = Varied(n=len(refs), table=t.ctypes.data if len(refs) else None, index=i.ctypes.data if len(refs) else None,
               values=_ptr(values))
    return v, (t, i, values)


_lib.trepb_last_error.restype = C.c_char_p
_lib.trepb_system_kernel_name.restype = C.c_char_p
_lib.trepb_specialized_name.restype = C.c_char_p
_lib.trepb_desc_hash.restype = C.c_uint64
_lib.trepb_struct_hash.restype = C.c_uint64
_lib.trepb_system_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
_lib.trepb_system_destroy.argtypes = [C.c_void_p]
_lib.trepb_system_destroy.restype = None
_lib.trepb_system_is_specialized.argtypes = [C.c_void_p]
_lib.trepb_system_is_cooperative.argtypes = [C.c_void_p]
_lib.trepb_system_kernel_name.argtypes = [C.c_void_p]
_lib.trepb_step_batch.argtypes = [C.c_void_p, C.POINTER(StepArgs)]
_lib.trepb_step_batch_dev.argtypes = [C.c_void_p, C.POINTER(StepArgs), C.c_void_p]
_lib.trepb_project_batch.argtypes = [C.c_void_p, C.POINTER(ProjectArgs)]
_lib.trepb_project_batch_dev.argtypes = [C.c_void_p, C.POINTER(ProjectArgs), C.c_void_p]
_lib.trepb_lqr_batch.argtypes = [C.c_int, C.POINTER(LqrArgs)]
_lib.trepb_lqr_batch_dev.argtypes = [C.c_int, C.POINTER(LqrArgs), C.c_void_p]
_lib.trepb_lq_batch.argtypes = [C.c_int, C.POINTER(LqArgs)]
_lib.trepb_lq_batch_dev.argtypes = [C.c_int, C.POINTER(LqArgs), C.c_void_p]
_lib.trepb_tangent_batch.argtypes = [C.c_int, C.POINTER(TangentArgs)]
_lib.trepb_tangent_batch_dev.argtypes = [C.c_int, C.POINTER(TangentArgs), C.c_void_p]
_lib.trepb_adjoint_batch.argtypes = [C.c_int, C.POINTER(AdjointArgs)]
_lib.trepb_adjoint_batch_dev.argtypes = [C.c_int, C.POINTER(AdjointArgs), C.c_void_p]
_lib.trepb_track_batch.argtypes = [C.c_int, C.POINTER(TrackArgs)]
_lib.trepb_track_batch_dev.argtypes = [C.c_int, C.POINTER(TrackArgs), C.c_void_p]
_lib.trepb_candidates_batch.argtypes = [C.c_int, C.POINTER(CandidatesArgs)]
_lib.trepb_candidates_batch_dev.argtypes = [C.c_int, C.POINTER(CandidatesArgs), C.c_void_p]
_lib.trepb_dare_batch.argtypes = [C.c_int, C.POINTER(DareArgs)]
_lib.trepb_dare_batch_dev.argtypes = [C.c_int, C.POINTER(DareArgs), C.c_void_p]
_lib.trepb_dlyap_batch.argtypes = [C.c_int, C.POINTER(DlyapArgs)]
_lib.trepb_dlyap_batch_dev.argtypes = [C.c_int, C.POINTER(DlyapArgs), C.c_void_p]
_lib.trepb_lqr_last_kernel_ms.argtypes = [C.c_int, C.POINTER(C.c_float)]
_lib.trepb_linearize_batch.argtypes = [C.c_void_p, C.POINTER(LinArgs)]
_lib.trepb_linearize_batch_dev.argtypes = [C.c_void_p, C.POINTER(LinArgs), C.c_void_p]
_lib.trepb_deriv2_batch.argtypes = [C.c_void_p, C.POINTER(D2Args)]
_lib.trepb_deriv2_batch_dev.argtypes = [C.c_void_p, C.POINTER(D2Args), C.c_void_p]
_lib.trepb_calc_p2_batch.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
_lib.trepb_calc_p2_batch_dev.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]
_lib.trepb_calc_f_batch.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_double] + [C.c_void_p] * 6
_lib.trepb_calc_f_batch_dev.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_double] + [C.c_void_p] * 7
_lib.trepb_discrete_fm2_batch.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_double] + [C.c_void_p] * 4
_lib.trepb_discrete_fm2_batch_dev.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_double] + [C.c_void_p] * 5
_lib.trepb_last_kernel_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
_lib.trepb_kernel_info.argtypes = [C.c_void_p, C.c_int] + [_ip] * 5
_lib.trepb_malloc.argtypes = [C.c_int, C.c_int64, C.POINTER(C.c_void_p)]
_lib.trepb_free.argtypes = [C.c_int, C.c_void_p]
_lib.trepb_host_alloc.argtypes = [C.c_int64, C.POINTER(C.c_void_p)]
_lib.trepb_host_free.argtypes = [C.c_void_p]
_lib.trepb_memcpy_h2d.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
_lib.trepb_memcpy_d2h.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
_lib.trepb_memset.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int64]
_lib.trepb_memcpy_d2d.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
_lib.trepb_comm_available.argtypes = [C.POINTER(C.c_int)]
_lib.trepb_comm_unique_id.argtypes = [C.c_char_p]
_lib.trepb_comm_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_char_p, C.POINTER(C.c_void_p)]
_lib.trepb_comm_destroy.argtypes = [C.c_void_p]
_lib.trepb_comm_destroy.restype = None
_lib.trepb_comm_rank.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
_lib.trepb_comm_allgather_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
_lib.trepb_comm_gather_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
_lib.trepb_ipc_export.argtypes = [C.c_int, C.c_void_p, C.c_char_p]
_lib.trepb_ipc_open.argtypes = [C.c_int, C.c_char_p, C.POINTER(C.c_void_p)]
_lib.trepb_ipc_close.argtypes = [C.c_int, C.c_void_p]
_lib.trepb_event_pair_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
_lib.trepb_event_record.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
_lib.trepb_event_elapsed_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
_lib.trepb_event_pair_destroy.argtypes = [C.c_void_p]
_lib.trepb_event_pair_destroy.restype = None
_lib.trepb_measure_fp64_peak.argtypes = [C.c_int, _dp]
_vp = C.POINTER(Varied)
_lib.trepb_varied_check.argtypes = [C.c_void_p, _vp]
# trepb_<call>_varied_batch[_dev]: the arguments of trepb_<call>_batch, then the trepb_varied (and the stream)
for _call in ("step", "project", "linearize", "calc_p2", "calc_f", "discrete_fm2", "deriv2"):
    _plain = getattr(_lib, "trepb_%s_batch" % _call).argtypes
    getattr(_lib, "trepb_%s_varied_batch" % _call).argtypes = _plain + [_vp]
    getattr(_lib, "trepb_%s_varied_batch_dev" % _call).argtypes = _plain + [_vp, C.c_void_p]
_lib.trepb_sincos_batch.argtypes = [C.c_int, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]

EXPORTS = [
    "trepb_abi_version", "trepb_last_error", "trepb_system_create", "trepb_system_destroy",
    "trepb_system_dims", "trepb_system_is_specialized", "trepb_system_is_cooperative", "trepb_system_kernel_name",
    "trepb_kernel_info", "trepb_validate", "trepb_codegen", "trepb_codegen_literal", "trepb_desc_hash", "trepb_struct_hash", "trepb_coop_dims",
    "trepb_num_specialized", "trepb_specialized_name", "trepb_step_batch", "trepb_step_batch_dev",
    "trepb_calc_p2_batch", "trepb_calc_p2_batch_dev", "trepb_calc_f_batch", "trepb_calc_f_batch_dev",
    "trepb_discrete_fm2_batch", "trepb_discrete_fm2_batch_dev", "trepb_project_batch", "trepb_project_batch_dev", "trepb_lqr_batch", "trepb_lqr_batch_dev", "trepb_lq_batch", "trepb_lq_batch_dev", "trepb_lqr_last_kernel_ms", "trepb_load_plugin", "trepb_linearize_batch",
    "trepb_linearize_batch_dev", "trepb_deriv2_batch", "trepb_deriv2_batch_dev", "trepb_device_count", "trepb_malloc", "trepb_free",
    "trepb_host_alloc", "trepb_host_free", "trepb_memset", "trepb_memcpy_h2d", "trepb_memcpy_d2h", "trepb_memcpy_d2d",
    "trepb_comm_available", "trepb_comm_unique_id", "trepb_comm_create", "trepb_comm_destroy", "trepb_comm_rank",
    "trepb_comm_allgather_dev", "trepb_comm_gather_dev", "trepb_ipc_export", "trepb_ipc_open", "trepb_ipc_close",
    "trepb_event_pair_create", "trepb_event_record", "trepb_event_elapsed_ms", "trepb_event_pair_destroy",
    "trepb_synchronize", "trepb_last_kernel_ms", "trepb_measure_fp64_peak", "trepb_sincos_batch",
    "trepb_varied_check", "trepb_step_varied_batch", "trepb_step_varied_batch_dev", "trepb_linearize_varied_batch",
    "trepb_linearize_varied_batch_dev", "trepb_project_varied_batch", "trepb_project_varied_batch_dev",
    "trepb_calc_p2_varied_batch", "trepb_calc_p2_varied_batch_dev", "trepb_calc_f_varied_batch",
    "trepb_calc_f_varied_batch_dev", "trepb_discrete_fm2_varied_batch", "trepb_discrete_fm2_varied_batch_dev",
    "trepb_deriv2_varied_batch", "trepb_deriv2_varied_batch_dev", "trepb_tangent_batch", "trepb_tangent_batch_dev",
    "trepb_adjoint_batch", "trepb_adjoint_batch_dev", "trepb_track_batch", "trepb_track_batch_dev",
    "trepb_candidates_batch", "trepb_candidates_batch_dev", "trepb_dare_batch", "trepb_dare_batch_dev",
    "trepb_dlyap_batch", "trepb_dlyap_batch_dev",
]


class TrepbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("trepb error %d: %s" % (code, msg))
        self.code = code


def _check(rc):
    if rc != 0:
        raise TrepbError(rc, (_lib.trepb_last_error() or b"").decode())


def raw():
    """The ctypes library object (for symbol checks)."""
    return _lib


def device_count():
    n = C.c_int(0)
    rc = _lib.trepb_device_count(C.byref(n))
    return n.value if rc == 0 else 0


def coop_dims(desc):
    """Shape the compile-time-size cooperative kernels are instantiated for: (nd, nk, nu, nc, links, points,
    chain pairs, levels, constrained dynamic configs, constrained configs, extras), or None when the cooperative
    kernels do not apply; extras = 1 for a system with LinearSprings / LinearDampers / spline springs / wrenches
    (their counts stay run-time data of the instantiation)."""
    cd, keep = D.to_c(desc)
    out = (C.c_int32 * 11)()
    if _lib.trepb_coop_dims(C.byref(cd), out) != 0:
        return None
    return tuple(out)


def lqr_raw(on_device, device, batch, nsteps, nX, nU, A, B, Q, R, Kfb, status, P0=None, q_per_step=False,
            r_per_step=False, stream=None):
    a = LqrArgs(batch=batch, nsteps=nsteps, nX=nX, nU=nU, q_per_step=1 if q_per_step else 0,
                r_per_step=1 if r_per_step else 0, A=_ptr(A), B=_ptr(B), Q=_ptr(Q), R=_ptr(R), Kfb=_ptr(Kfb),
                P0=_ptr(P0), status=_ptr(status))
    if on_device:
        _check(_lib.trepb_lqr_batch_dev(device, C.byref(a), stream))
    else:
        _check(_lib.trepb_lqr_batch(device, C.byref(a)))


def load_plugin(path):
    """Load a plug-in of specialised kernels (trep_b200.build.build_plugin); returns the number of kernel sets it added."""
    _lib.trepb_load_plugin.argtypes = [C.c_char_p, C.POINTER(C.c_int)]
    n = C.c_int(0)
    _check(_lib.trepb_load_plugin(os.fspath(path).encode(), C.byref(n)))
    return int(n.value)


def specialize(desc, kind="auto", ext=False, verbose=False):
    """Builds (once per structure: the library is named by trepb_struct_hash and rebuilt only when older than the
    headers) and loads a plug-in of kernels compiled for `desc`'s structure, so that System(desc) - and every other
    description with the same structure, whatever its masses, lengths and gains - runs on them instead of the
    table-driven kernels.  kind / ext as trep_b200.build.build_plugin.  Needs nvcc (a minute per structure); raises
    RuntimeError without it: there is no silent fallback.  Returns the number of kernel sets added (0 if this
    structure's plug-in was already loaded)."""
    import shutil
    from . import build
    if kind == "auto":
        kind = "thread" if desc.nd + desc.nk <= 6 else "coop"
    name = "s%016x_%s%s" % (struct_hash(desc), kind, "_ext" if ext else "")
    if name in _specialized:
        return 0
    if shutil.which(build.NVCC) is None:
        raise RuntimeError("trep_b200.lib.specialize needs nvcc (%s) to build the plug-in" % build.NVCC)
    n = load_plugin(build.build_plugin(desc, name, verbose=verbose, kind=kind, ext=ext))
    _specialized.add(name)
    return n


_specialized = set()


def lqr_last_kernel_ms(device=0):
    """Device time (CUDA events) of the last Riccati kernel launched on `device`."""
    ms = C.c_float()
    _check(_lib.trepb_lqr_last_kernel_ms(device, C.byref(ms)))
    return float(ms.value)


def solve_tv_lqr(A, B, Q, R, device=0):
    """Batched discopt.dlqr.solve_tv_lqr (trep/discopt/dlqr.py:9-38) on the GPU.
    A [R,K,nX,nX] or [K,nX,nX]; B likewise; Q [nX,nX] or [K+1,nX,nX]; R [nU,nU] or [K,nU,nU].
    Returns (K [..,K,nU,nX], P0 [..,nX,nX])."""
    A = np.ascontiguousarray(np.asarray(A, float)); B = np.ascontiguousarray(np.asarray(B, float))
    single = A.ndim == 3
    if single:
        A, B = A[None], B[None]
    Rn, K, nX = A.shape[0], A.shape[1], A.shape[2]
    nU = B.shape[3]
    Q = np.ascontiguousarray(np.asarray(Q, float)); R = np.ascontiguousarray(np.asarray(R, float))
    Kfb = np.zeros((Rn, K, nU, nX)); P0 = np.zeros((Rn, nX, nX)); status = np.zeros(Rn, np.int32)
    lqr_raw(False, device, Rn, K, nX, nU, A, B, Q, R, Kfb, status, P0=P0, q_per_step=Q.ndim == 3, r_per_step=R.ndim == 3)
    if np.any(status != 0):
        raise TrepbError(0, "singular gamma in the Riccati sweep of rollout(s) %s" % np.flatnonzero(status != 0)[:8])
    return (Kfb[0], P0[0]) if single else (Kfb, P0)


def lq_raw(on_device, device, batch, nsteps, nX, nU, A, B, Q, S, R, q, r, Kfb, Cff, status, P0=None, b0=None,
           cost_per_rollout=False, stream=None):
    a = LqArgs(batch=batch, nsteps=nsteps, nX=nX, nU=nU, cost_per_rollout=1 if cost_per_rollout else 0,
               A=_ptr(A), B=_ptr(B), Q=_ptr(Q), S=_ptr(S), R=_ptr(R), q=_ptr(q), r=_ptr(r), Kfb=_ptr(Kfb),
               C=_ptr(Cff), P0=_ptr(P0), b0=_ptr(b0), status=_ptr(status))
    if on_device:
        _check(_lib.trepb_lq_batch_dev(device, C.byref(a), stream))
    else:
        _check(_lib.trepb_lq_batch(device, C.byref(a)))


def solve_tv_lq(A, B, q, r, Q, S, R, device=0):
    """Batched discopt.dlqr.solve_tv_lq (trep/discopt/dlqr.py:41-81) on the GPU.
    One rollout: A [K,nX,nX], B [K,nX,nU], q [K+1,nX], r [K,nU], Q [K+1,nX,nX], S [K,nX,nU] or None,
    R [K,nU,nU]; a batch: one more leading axis on A and B, and either the same on every cost array
    (one cost per rollout) or none (costs shared).  Returns (K, C, P0, b0)."""
    f = lambda x: np.ascontiguousarray(np.asarray(x, float))
    A, B, q, r, Q, R = f(A), f(B), f(q), f(r), f(Q), f(R)
    S = None if S is None else f(S)
    single = A.ndim == 3
    if single:
        A, B = A[None], B[None]
    Rn, K, nX = A.shape[0], A.shape[1], A.shape[2]
    nU = B.shape[3]
    per = Q.ndim == 4
    Kfb = np.zeros((Rn, K, nU, nX)); Cff = np.zeros((Rn, K, nU)); P0 = np.zeros((Rn, nX, nX)); b0 = np.zeros((Rn, nX))
    status = np.zeros(Rn, np.int32)
    lq_raw(False, device, Rn, K, nX, nU, A, B, Q, S, R, q, r, Kfb, Cff, status, P0=P0, b0=b0, cost_per_rollout=per)
    if np.any(status != 0):
        raise TrepbError(0, "singular gamma in the Riccati sweep of rollout(s) %s" % np.flatnonzero(status != 0)[:8])
    return (Kfb[0], Cff[0], P0[0], b0[0]) if single else (Kfb, Cff, P0, b0)


DARE_OK, DARE_NOT_CONVERGED, DARE_SINGULAR, DARE_NONFINITE = 0, -1, -2, -3   # TREPB_DARE_* (trepb.h)
DARE_STATUS = {DARE_NOT_CONVERGED: "not converged", DARE_SINGULAR: "singular R, I + G H or R + B^T P B",
               DARE_NONFINITE: "non-finite iterate (no stabilizing solution?)"}


def dare_raw(on_device, device, batch, nX, nU, A, B, Q, R, status, K=None, P=None, S=None, iterations=None,
             q_per_rollout=False, r_per_rollout=False, s_per_rollout=False, tol=1e-13, max_iterations=64, stream=None):
    """trepb_dare_batch[_dev]: the stationary LQR gain K [batch,nU,nX] (u = -K x) and the stabilizing DARE solution
    P [batch,nX,nX] of `batch` models A [batch,nX,nX], B [batch,nX,nU]; Q / R / S one matrix or one per model."""
    a = DareArgs(batch=batch, nX=nX, nU=nU, max_iterations=max_iterations, q_per_rollout=1 if q_per_rollout else 0,
                 r_per_rollout=1 if r_per_rollout else 0, s_per_rollout=1 if s_per_rollout else 0, tol=tol,
                 A=_ptr(A), B=_ptr(B), Q=_ptr(Q), R=_ptr(R), S=_ptr(S), K=_ptr(K), P=_ptr(P), status=_ptr(status),
                 iterations=_ptr(iterations))
    if on_device:
        _check(_lib.trepb_dare_batch_dev(device, C.byref(a), stream))
    else:
        _check(_lib.trepb_dare_batch(device, C.byref(a)))


def solve_dare(A, B, Q, R, S=None, tol=1e-13, max_iterations=64, device=0):
    """Stationary discrete LQR on the GPU: the stabilizing solution P of
        P = A^T P A - (A^T P B + S)(R + B^T P B)^-1 (B^T P A + S^T) + Q
    (scipy.linalg.solve_discrete_are(A, B, Q, R, s=S)) and K = (R + B^T P B)^-1 (B^T P A + S^T), u = -K x.
    One problem: A [nX,nX], B [nX,nU], Q [nX,nX], R [nU,nU], S [nX,nU] or None; a batch: one more leading axis on A and
    B, and on each of Q / R / S either the same (one per model) or none (shared).  Returns (K, P, status, iterations);
    a single problem whose status is not DARE_OK raises TrepbError."""
    f = lambda x: None if x is None else np.ascontiguousarray(np.asarray(x, float))
    A, B, Q, R, S = f(A), f(B), f(Q), f(R), f(S)
    single = A.ndim == 2
    if single:
        A, B = A[None], B[None]
    Rn, nX, nU = A.shape[0], A.shape[1], B.shape[2]
    K, P = np.zeros((Rn, nU, nX)), np.zeros((Rn, nX, nX))
    status, iters = np.zeros(Rn, np.int32), np.zeros(Rn, np.int32)
    dare_raw(False, device, Rn, nX, nU, A, B, Q, R, status, K=K, P=P, S=S, iterations=iters,
             q_per_rollout=Q.ndim == 3, r_per_rollout=R.ndim == 3, s_per_rollout=S is not None and S.ndim == 3,
             tol=tol, max_iterations=max_iterations)
    if single:
        if status[0] != DARE_OK:
            raise TrepbError(0, "DARE failed after %d doubling steps: %s (status %d)"
                             % (iters[0], DARE_STATUS.get(int(status[0]), "?"), status[0]))
        return K[0], P[0], int(status[0]), int(iters[0])
    return K, P, status, iters


DLYAP_STABLE, DLYAP_NOT_CONVERGED, DLYAP_NONFINITE, DLYAP_BAD_INDEX = 0, -1, -3, -4   # TREPB_DLYAP_* (trepb.h)
DLYAP_STATUS = {DLYAP_STABLE: "stable", DLYAP_NOT_CONVERGED: "not converged (rho(A - B K) >= 1?)",
                DLYAP_NONFINITE: "non-finite iterate (unstable closed loop)",
                DLYAP_BAD_INDEX: "gain or model index out of range"}


def dlyap_raw(on_device, device, pairs, gains, models, nX, nU, A, B, K, Q, R, status, S=None, gain_index=None,
              model_index=None, x0=None, W=None, P=None, cost=None, iterations=None, q_per_model=False,
              r_per_model=False, s_per_model=False, x0_per_pair=False, tol=1e-13, max_iterations=64, stream=None):
    """trepb_dlyap_batch[_dev]: for pair p, gain K[gain_index[p]] [nU,nX] (u = -K x) under model
    A[model_index[p]] [nX,nX], B[model_index[p]] [nX,nU] (either index None: gain p / model p), the closed-loop
    cost-to-go P [pairs,nX,nX] of P = A_c^T P A_c + Q_c, cost [pairs] = x0^T P x0 or trace(P W), and the stability
    verdict status [pairs] (DLYAP_*); Q / R / S one matrix or one per model."""
    a = DlyapArgs(pairs=pairs, gains=gains, models=models, nX=nX, nU=nU, max_iterations=max_iterations,
                  q_per_model=1 if q_per_model else 0, r_per_model=1 if r_per_model else 0,
                  s_per_model=1 if s_per_model else 0, x0_per_pair=1 if x0_per_pair else 0, tol=tol,
                  A=_ptr(A), B=_ptr(B), K=_ptr(K), Q=_ptr(Q), R=_ptr(R), S=_ptr(S), gain_index=_ptr(gain_index),
                  model_index=_ptr(model_index), x0=_ptr(x0), W=_ptr(W), P=_ptr(P), cost=_ptr(cost),
                  status=_ptr(status), iterations=_ptr(iterations))
    if on_device:
        _check(_lib.trepb_dlyap_batch_dev(device, C.byref(a), stream))
    else:
        _check(_lib.trepb_dlyap_batch(device, C.byref(a)))


def solve_closed_loop(A, B, K, Q, R, S=None, x0=None, W=None, gain_index=None, model_index=None, tol=1e-13,
                      max_iterations=64, device=0):
    """Closed-loop cost and stability of stationary gains on the GPU: for u = -K x under x+ = A x + B u, the solution
    P of P = A_c^T P A_c + Q_c with A_c = A - B K and Q_c = Q - S K - K^T S^T + K^T R K
    (scipy.linalg.solve_discrete_lyapunov(A_c.T, Q_c)), the infinite-horizon cost of the stage cost
    x^T Q x + 2 x^T S u + u^T R u, which exists exactly when rho(A_c) < 1.
    One problem: A [nX,nX], B [nX,nU], K [nU,nX].  A batch: A [M,nX,nX], B [M,nX,nU], K [G,nU,nX], and pair p
    evaluates gain gain_index[p] under model model_index[p] (either None: gain p / model p; without both, G = M
    pairs).  Q / R / S shared or one per model (leading axis M).  cost = x0^T P x0 (x0 [nX], or [pairs,nX] one per
    pair) or trace(P W) (W [nX,nX]); None without either.  Returns (P, cost, status, iterations); the cost of a pair
    that is not DLYAP_STABLE is +inf.  A single problem whose status is not DLYAP_STABLE raises TrepbError."""
    f = lambda x: None if x is None else np.ascontiguousarray(np.asarray(x, float))
    A, B, K, Q, R, S, x0, W = f(A), f(B), f(K), f(Q), f(R), f(S), f(x0), f(W)
    single = A.ndim == 2
    if single:
        A, B, K = A[None], B[None], K[None]
    M, nX, nU, G = A.shape[0], A.shape[1], B.shape[2], K.shape[0]
    idx = lambda i: None if i is None else np.ascontiguousarray(np.asarray(i, dtype=np.int32).ravel())
    gain_index, model_index = idx(gain_index), idx(model_index)
    if gain_index is not None:
        pairs = gain_index.size
    elif model_index is not None:
        pairs = model_index.size
    elif G == M:
        pairs = G
    else:
        raise ValueError("%d gains and %d models: pass gain_index / model_index" % (G, M))
    if gain_index is not None and model_index is not None and model_index.size != pairs:
        raise ValueError("gain_index has %d pairs, model_index %d" % (pairs, model_index.size))
    P = np.zeros((pairs, nX, nX))
    cost = np.zeros(pairs) if x0 is not None or W is not None else None
    status, iters = np.zeros(pairs, np.int32), np.zeros(pairs, np.int32)
    dlyap_raw(False, device, pairs, G, M, nX, nU, A, B, K, Q, R, status, S=S, gain_index=gain_index,
              model_index=model_index, x0=x0, W=W, P=P, cost=cost, iterations=iters, q_per_model=Q.ndim == 3,
              r_per_model=R.ndim == 3, s_per_model=S is not None and S.ndim == 3,
              x0_per_pair=x0 is not None and x0.ndim == 2, tol=tol, max_iterations=max_iterations)
    if single:
        if status[0] != DLYAP_STABLE:
            raise TrepbError(0, "closed-loop Lyapunov solve failed after %d doubling steps: %s (status %d)"
                             % (iters[0], DLYAP_STATUS.get(int(status[0]), "?"), status[0]))
        return P[0], None if cost is None else float(cost[0]), int(status[0]), int(iters[0])
    return P, cost, status, iters


def tangent_raw(on_device, device, batch, nsteps, nX, nU, A, B, K, dX, dU, bdX=None, bdU=None, x0=None, stream=None):
    a = TangentArgs(batch=batch, nsteps=nsteps, nX=nX, nU=nU, A=_ptr(A), B=_ptr(B), K=_ptr(K), bdX=_ptr(bdX),
                    bdU=_ptr(bdU), x0=_ptr(x0), dX=_ptr(dX), dU=_ptr(dU))
    if on_device:
        _check(_lib.trepb_tangent_batch_dev(device, C.byref(a), stream))
    else:
        _check(_lib.trepb_tangent_batch(device, C.byref(a)))


def adjoint_raw(on_device, device, batch, nsteps, nX, nU, A, B, m_dx, z, K=None, l_dx=None, l_du=None, z1=None,
                stream=None):
    a = AdjointArgs(batch=batch, nsteps=nsteps, nX=nX, nU=nU, A=_ptr(A), B=_ptr(B), K=_ptr(K), l_dx=_ptr(l_dx),
                    l_du=_ptr(l_du), m_dx=_ptr(m_dx), z=_ptr(z), z1=_ptr(z1))
    if on_device:
        _check(_lib.trepb_adjoint_batch_dev(device, C.byref(a), stream))
    else:
        _check(_lib.trepb_adjoint_batch(device, C.byref(a)))


def _sweep_in(A, B, single, *more):
    """float64 contiguous copies, a leading rollout axis added to a single trajectory's arrays (None stays None)."""
    f = lambda x: None if x is None else np.ascontiguousarray(np.asarray(x, float))
    out = [f(x) for x in (A, B) + more]
    return [None if x is None else (x[None] if single else x) for x in out]


def tangent_sweep(A, B, K, bdX, bdU, x0=None, device=0):
    """Batched DSystem.dproject (trep/discopt/dsystem.py:460-471) on the GPU:
    dX[0] = x0 (default bdX[0]); dU[k] = bdU[k] - K[k] (dX[k] - bdX[k]); dX[k+1] = A[k] dX[k] + B[k] dU[k].
    One trajectory: A [K,nX,nX], B [K,nX,nU], K [K,nU,nX], bdX [K+1,nX], bdU [K,nU], x0 [nX]; a batch: one more
    leading axis on every array.  bdX / bdU / x0 may be None (zero; x0 then defaults to bdX[0]).
    Returns (dX, dU)."""
    A = np.asarray(A)
    single = A.ndim == 3
    A, B, K, bdX, bdU, x0 = _sweep_in(A, B, single, K, bdX, bdU, x0)
    Rn, n, nX = A.shape[0], A.shape[1], A.shape[2]
    nU = B.shape[3]
    dX, dU = np.zeros((Rn, n + 1, nX)), np.zeros((Rn, n, nU))
    tangent_raw(False, device, Rn, n, nX, nU, A, B if nU else None, K if nU else None, dX, dU if nU else None,
                bdX=bdX, bdU=bdU if nU else None, x0=x0)
    return (dX[0], dU[0]) if single else (dX, dU)


def adjoint_sweep(A, B, m_dx, l_dx=None, l_du=None, K=None, device=0):
    """The costate recursion of DOptimizer.calc_newton_model (trep/discopt/doptimizer.py:319-345) on the GPU:
    z[K] = m_dx; z[k] = l_dx[k] - K[k]^T l_du[k] + (A[k] - B[k] K[k])^T z[k+1] (K None: z[k] = l_dx[k] + A[k]^T z[k+1]).
    One trajectory: A [K,nX,nX], B [K,nX,nU], m_dx [nX], l_dx [K,nX], l_du [K,nU], K [K,nU,nX]; a batch: one more
    leading axis on every array.  l_dx / l_du may be None (zero).  Returns z [..,K+1,nX]."""
    A = np.asarray(A)
    single = A.ndim == 3
    A, B, m_dx, l_dx, l_du, K = _sweep_in(A, B, single, m_dx, l_dx, l_du, K)
    Rn, n, nX = A.shape[0], A.shape[1], A.shape[2]
    nU = B.shape[3]
    z = np.zeros((Rn, n + 1, nX))
    adjoint_raw(False, device, Rn, n, nX, nU, A, B if nU else None, m_dx, z, K=K if nU else None, l_dx=l_dx,
                l_du=l_du if nU else None)
    return z[0] if single else z


TRACK_OUTPUTS = ("cost", "dcost", "q", "r", "l_dx", "m_dx", "Qm", "Sm", "Rm")


def track_raw(on_device, device, batch, nsteps, nX, nU, nref=1, stream=None, **arrays):
    """trepb_track_batch[_dev]: arrays by field name of trepb_track_args (X, U, Xd, Ud, Q, R, ref_index, dX, dU, fdxdx,
    fdxdu, fdudu and the outputs TRACK_OUTPUTS); missing ones are NULL."""
    a = TrackArgs(batch=batch, nsteps=nsteps, nX=nX, nU=nU, nref=nref)
    for n, v in arrays.items():
        setattr(a, n, _ptr(v))
    if on_device:
        _check(_lib.trepb_track_batch_dev(device, C.byref(a), stream))
    else:
        _check(_lib.trepb_track_batch(device, C.byref(a)))


def candidates_raw(on_device, device, groups, ncand, nsteps, nX, nU, lam, X, U, dX, dU, Kproj, bX, bU, Kc, rows=None,
                   nrollouts=0, stream=None):
    a = CandidatesArgs(groups=groups, ncand=ncand, nsteps=nsteps, nX=nX, nU=nU, nrollouts=nrollouts, rows=_ptr(rows),
                       lam=_ptr(lam), X=_ptr(X), U=_ptr(U), dX=_ptr(dX), dU=_ptr(dU), Kproj=_ptr(Kproj), bX=_ptr(bX),
                       bU=_ptr(bU), Kc=_ptr(Kc))
    if on_device:
        _check(_lib.trepb_candidates_batch_dev(device, C.byref(a), stream))
    else:
        _check(_lib.trepb_candidates_batch(device, C.byref(a)))


def track_cost(X, U, Xd, Ud, Q, R, ref_index=None, dX=None, dU=None, newton=None, outputs=TRACK_OUTPUTS, device=0):
    """The tracking cost of DCost (trep/discopt/dcost.py) and its LQ model on the GPU (trepb_track_batch).
    X [B,K+1,nX], U [B,K,nU]; Xd [K+1,nX] / Ud [K,nU] (one reference) or [nref,..] with ref_index [B] naming each
    trajectory's reference; Q [nX,nX], R [nU,nU]; dX / dU as X / U for dcost; newton = (fdxdx [B,K,nX,nX], fdxdu
    [B,K,nX,nU], fdudu [B,K,nU,nU]) added to the model.  Returns a dict of the requested outputs (cost and dcost [B],
    q [B,K+1,nX], r [B,K,nU], l_dx [B,K,nX], m_dx [B,nX], Qm [B,K+1,nX,nX], Sm [B,K,nX,nU], Rm [B,K,nU,nU]); dcost
    only when dX is given."""
    f = lambda x: None if x is None else np.ascontiguousarray(np.asarray(x, float))
    X, U, Xd, Ud, Q, R, dX, dU = (f(x) for x in (X, U, Xd, Ud, Q, R, dX, dU))
    Bn, K, nX = X.shape[0], X.shape[1] - 1, X.shape[2]
    nU = U.shape[2]
    if Xd.ndim == 2:
        Xd, Ud = Xd[None], Ud[None]
    shapes = dict(cost=(Bn,), dcost=(Bn,), q=(Bn, K + 1, nX), r=(Bn, K, nU), l_dx=(Bn, K, nX), m_dx=(Bn, nX),
                  Qm=(Bn, K + 1, nX, nX), Sm=(Bn, K, nX, nU), Rm=(Bn, K, nU, nU))
    out = {n: np.zeros(shapes[n]) for n in outputs if n != "dcost" or dX is not None}
    arrays = dict(X=X, U=U, Xd=Xd, Ud=Ud, Q=Q, R=R, dX=dX, dU=dU)
    if ref_index is not None:
        arrays["ref_index"] = np.ascontiguousarray(ref_index, dtype=np.int32)
    if newton is not None:
        arrays.update(zip(("fdxdx", "fdxdu", "fdudu"), (f(x) for x in newton)))
    if nU == 0:
        arrays = {n: v for n, v in arrays.items() if n not in ("U", "Ud", "R", "dU", "fdxdu", "fdudu")}
    arrays.update({n: v for n, v in out.items() if nU or n not in ("r", "Sm", "Rm")})
    track_raw(False, device, Bn, K, nX, nU, nref=Xd.shape[0], **arrays)
    return out


def specialized_names():
    return [_lib.trepb_specialized_name(i).decode() for i in range(_lib.trepb_num_specialized())]


def desc_hash(desc):
    cd, keep = D.to_c(desc)
    return int(_lib.trepb_desc_hash(C.byref(cd)))


def struct_hash(desc):
    """Hash of the structure only (what a specialised kernel is compiled for); see include/trepb.h."""
    cd, keep = D.to_c(desc)
    return int(_lib.trepb_struct_hash(C.byref(cd)))


def validate(desc):
    cd, keep = D.to_c(desc)
    _check(_lib.trepb_validate(C.byref(cd)))


def check_params(desc, refs):
    """Raises TrepbError (TREPB_ERR_INVALID, the entry named) unless every SystemDesc.param_ref in `refs` may vary
    per instance (trepb_varied_check: non-zero, not +-1 in frame_se3, not a spline x-point, no repeats)."""
    cd, keep = D.to_c(desc)
    v, vkeep = _varied((refs, None))
    _check(_lib.trepb_varied_check(C.byref(cd), C.byref(v)))


def measure_fp64_peak(device=0):
    v = C.c_double(0)
    _check(_lib.trepb_measure_fp64_peak(device, C.byref(v)))
    return v.value


def sincos(x, device=0):
    """(sin, cos) of an array as the kernels compute them (diagnostic)."""
    x = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
    s, c = np.empty_like(x), np.empty_like(x)
    _check(_lib.trepb_sincos_batch(device, x.size, x.ctypes.data, s.ctypes.data, c.ctypes.data))
    return s, c


def synchronize(device=0):
    _check(_lib.trepb_synchronize(device))


class EventTimer:
    """CUDA-event pair on a stream (trepb_event_*): `with EventTimer(dev) as t: ...launches...; t.ms`."""

    def __init__(self, device=0, stream=None):
        self.device, self.stream = device, stream
        self._h = C.c_void_p()
        _check(_lib.trepb_event_pair_create(device, C.byref(self._h)))
        self.ms = None

    def __enter__(self):
        _check(_lib.trepb_event_record(self._h, 0, self.stream))
        return self

    def __exit__(self, *exc):
        _check(_lib.trepb_event_record(self._h, 1, self.stream))
        v = C.c_float(0)
        _check(_lib.trepb_event_elapsed_ms(self._h, C.byref(v)))
        self.ms = v.value
        return False

    def __del__(self):
        try:
            if self._h:
                _lib.trepb_event_pair_destroy(self._h)
                self._h = None
        except Exception:
            pass


class DeviceBuffer:
    """HBM buffer owned through the C ABI (so that a host without torch can drive the library)."""

    def __init__(self, device, shape, dtype=np.float64):
        self.device, self.shape, self.dtype = device, tuple(shape), np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        p = C.c_void_p()
        _check(_lib.trepb_malloc(device, self.nbytes, C.byref(p)))
        self.ptr = p.value

    def data_ptr(self):
        return self.ptr

    def upload(self, host):
        host = np.ascontiguousarray(host, dtype=self.dtype)
        assert host.nbytes == self.nbytes, (host.shape, self.shape)
        _check(_lib.trepb_memcpy_h2d(self.device, self.ptr, host.ctypes.data, self.nbytes))
        return self

    def download(self, out=None):
        if out is None:
            out = np.empty(self.shape, self.dtype)
        _check(_lib.trepb_memcpy_d2h(self.device, out.ctypes.data, self.ptr, self.nbytes))
        return out

    def download_row(self, i):
        """Element i of the first axis, as an array of shape shape[1:]."""
        out = np.empty(self.shape[1:], self.dtype)
        _check(_lib.trepb_memcpy_d2h(self.device, out.ctypes.data, self.ptr + i * out.nbytes, out.nbytes))
        return out

    def zero(self):
        _check(_lib.trepb_memset(self.device, self.ptr, 0, self.nbytes))
        return self

    def free(self):
        if self.ptr:
            _lib.trepb_free(self.device, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def pinned_empty(shape, dtype=np.float64):
    """numpy array backed by pinned host memory (cudaHostAlloc) for the end-to-end path."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
    p = C.c_void_p()
    _check(_lib.trepb_host_alloc(max(n, 1), C.byref(p)))
    buf = (C.c_char * max(n, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)
    return arr


def _ptr(x):
    """Address of a numpy array / DeviceBuffer / torch tensor, or None."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    return x.data_ptr()


# trepb_system_create flag: per-instance parameters on a cooperative handle (trepb.h)
FLAG_COOP_VARIED = 128


class System:
    """Handle of a flattened system resident on one GPU (trepb_system)."""

    def __init__(self, desc: D.SystemDesc, device=0, specialize=True, cooperative=None, d2_pairwise=False, literal=True,
                 coop_one_warp=False, coop_two_warps=False, coop_varied=False):
        """specialize=False: skip the ahead-of-time specialised kernels.  cooperative: None = let
        the library choose between one thread and one warp per instance for a table-driven system,
        False = always one thread, True = always the cooperative kernels (their compile-time-size
        flavour when one was built for this shape, unless specialize=False).  d2_pairwise: second
        derivatives of a table-driven system by one hyper-dual residual evaluation per parameter
        pair instead of one dual evaluation of the Jacobian tables per parameter.  coop_one_warp /
        coop_two_warps: for shapes whose cooperative kernels were built in several flavours, the one-warp
        flavour with the whole workspace in shared memory / the two-warps-per-instance flavour instead of
        the default (TREPB_FLAG_COOP_ONE_WARP, TREPB_FLAG_COOP_TWO_WARPS).  coop_varied: on a cooperative handle,
        per-instance parameters (params=...) run on the varied cooperative kernels instead of being refused
        (TREPB_FLAG_COOP_VARIED); it changes nothing else."""
        self.desc = desc
        self.device = device
        cd, self._keep = D.to_c(desc)
        h = C.c_void_p()
        flags = 0 if specialize else 1
        if cooperative is False:
            flags |= 2
        elif cooperative is True:
            flags |= 4
        if d2_pairwise:
            flags |= 8
        if coop_one_warp:
            flags |= 32
        if coop_two_warps:
            flags |= 64
        if coop_varied:
            flags |= FLAG_COOP_VARIED
        if not literal:
            flags |= 16     # skip an all-literal instantiation: the run-time-parameter kernel of the structure
        _check(_lib.trepb_system_create(C.byref(cd), device, flags, C.byref(h)))
        self._h = h
        self.nq, self.nd, self.nk, self.nu, self.nc = desc.nq, desc.nd, desc.nk, desc.nu, desc.nc
        self.nX, self.nU = desc.nX, desc.nU

    @property
    def specialized(self):
        return bool(_lib.trepb_system_is_specialized(self._h))

    @property
    def cooperative(self):
        return bool(_lib.trepb_system_is_cooperative(self._h))

    @property
    def kernel_name(self):
        return _lib.trepb_system_kernel_name(self._h).decode()

    def kernel_info(self, which):
        v = [C.c_int32(0) for _ in range(5)]
        _check(_lib.trepb_kernel_info(self._h, which, *[C.byref(x) for x in v]))
        return dict(zip(["regs", "local_bytes", "blocks_per_sm", "block", "smem_bytes"], [x.value for x in v]))

    def last_kernel_ms(self):
        ms = C.c_float(0)
        _check(_lib.trepb_last_kernel_ms(self._h, C.byref(ms)))
        return ms.value

    def close(self):
        if getattr(self, "_h", None):
            _lib.trepb_system_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- raw calls: every array argument is a pointer-like (numpy => host entry point,
    #      anything with data_ptr() => device entry point); the caller owns shapes/dtypes ----------
    def _call(self, call, on_device, params, stream, *args):
        """trepb_<call>[_varied]_batch[_dev](handle, *args[, varied][, stream])."""
        tail = []
        if params is not None:
            v, keep = _varied(params)   # keep: the arrays v points into, alive until the call returns
            tail.append(C.byref(v))
        if on_device:
            tail.append(stream)
        name = "trepb_%s%s_batch%s" % (call, "" if params is None else "_varied", "_dev" if on_device else "")
        _check(getattr(_lib, name)(self._h, *args, *tail))

    def step_raw(self, on_device, batch, nsteps, t0, dt, q1, p1, u1, k2, q2_guess, lambda_guess,
                 q2, p2, lambda1, iters, status, tolerance=1e-10, max_iterations=200,
                 sample_every=0, traj_q=None, traj_p=None, stream=None, times=None, params=None):
        """params: None, or (refs, values [B][len(refs)]) per-instance parameters (trepb_step_varied_batch*)."""
        a = StepArgs(times=_ptr(times), batch=batch, nsteps=nsteps, max_iterations=max_iterations, t0=t0, dt=dt,
                     tolerance=tolerance, q1=_ptr(q1), p1=_ptr(p1), u1=_ptr(u1), k2=_ptr(k2),
                     q2_guess=_ptr(q2_guess), lambda_guess=_ptr(lambda_guess), q2=_ptr(q2),
                     p2=_ptr(p2), lambda1=_ptr(lambda1), iters=_ptr(iters), status=_ptr(status),
                     sample_every=sample_every, traj_q=_ptr(traj_q), traj_p=_ptr(traj_p))
        self._call("step", on_device, params, stream, C.byref(a))

    @staticmethod
    def _lin_args(batch, q1, p1, u1, k2, status, t1=None, t2=None, t1_scalar=0.0, dt_scalar=0.0,
                  q2_guess=None, lambda_guess=None, q2=None, p2=None, lambda1=None, iters=None,
                  A=None, B=None, raw=None, tolerance=1e-10, max_iterations=200, traj_len=0):
        a = LinArgs(traj_len=traj_len, batch=batch, max_iterations=max_iterations, tolerance=tolerance, t1=_ptr(t1),
                    t2=_ptr(t2), t1_scalar=t1_scalar, dt_scalar=dt_scalar, q1=_ptr(q1), p1=_ptr(p1),
                    u1=_ptr(u1), k2=_ptr(k2), q2_guess=_ptr(q2_guess),
                    lambda_guess=_ptr(lambda_guess), q2=_ptr(q2), p2=_ptr(p2),
                    lambda1=_ptr(lambda1), iters=_ptr(iters), status=_ptr(status), A=_ptr(A), B=_ptr(B))
        for n, v in (raw or {}).items():
            setattr(a, n, _ptr(v))
        return a

    def linearize_raw(self, on_device, batch, q1, p1, u1, k2, status, stream=None, params=None, **kw):
        """params: None, or (refs, values) with one row per instance, or per trajectory when traj_len >= 2."""
        a = self._lin_args(batch, q1, p1, u1, k2, status, **kw)
        self._call("linearize", on_device, params, stream, C.byref(a))

    def deriv2_raw(self, on_device, batch, q1, p1, u1, k2, status, d2, stream=None, z=None,
                   fdxdx=None, fdxdu=None, fdudu=None, params=None, **kw):
        """d2: {"q2_dq1dq1": array, ...} any subset of D2_WHICH x D2_KINDS; z + fdxdx/fdxdu/fdudu:
        the z-contracted forms of DSystem.fdxdx(z) / fdxdu(z) / fdudu(z).  params: None, or (refs, values) with one
        row per instance (trepb_deriv2_varied_batch*)."""
        a = D2Args()
        a.lin = self._lin_args(batch, q1, p1, u1, k2, status, **kw)
        a.z, a.fdxdx, a.fdxdu, a.fdudu = _ptr(z), _ptr(fdxdx), _ptr(fdxdu), _ptr(fdudu)
        for n, v in d2.items():
            w, kd = n.split("_")
            a.d2[10 * D2_WHICH.index(w) + D2_KINDS.index(kd)] = _ptr(v)
        self._call("deriv2", on_device, params, stream, C.byref(a))

    def project_raw(self, on_device, batch, nsteps, t0, dt, bX, bU, Kfb, X, U, status, k_per_instance=False,
                    use_hint=True, iters=None, fail_step=None, tolerance=1e-10, max_iterations=200, stream=None,
                    times=None, params=None):
        a = ProjectArgs(times=_ptr(times), batch=batch, nsteps=nsteps, max_iterations=max_iterations, t0=t0, dt=dt, tolerance=tolerance,
                        bX=_ptr(bX), bU=_ptr(bU), Kfb=_ptr(Kfb), k_per_instance=1 if k_per_instance else 0,
                        use_hint=1 if use_hint else 0, X=_ptr(X), U=_ptr(U), iters=_ptr(iters), status=_ptr(status),
                        fail_step=_ptr(fail_step))
        self._call("project", on_device, params, stream, C.byref(a))

    def calc_p2_raw(self, on_device, batch, dt, q0, q1, p, stream=None, params=None):
        self._call("calc_p2", on_device, params, stream, batch, dt, _ptr(q0), _ptr(q1), _ptr(p))

    def calc_f_raw(self, on_device, batch, t1, t2, q1, q2, p1, u1, lambda1, f, stream=None, params=None):
        self._call("calc_f", on_device, params, stream, batch, t1, t2, _ptr(q1), _ptr(q2), _ptr(p1), _ptr(u1),
                   _ptr(lambda1), _ptr(f))

    def discrete_fm2_raw(self, on_device, batch, t1, t2, q1, q2, u1, fm2, stream=None, params=None):
        self._call("discrete_fm2", on_device, params, stream, batch, t1, t2, _ptr(q1), _ptr(q2), _ptr(u1), _ptr(fm2))

    # ---- numpy convenience (host entry points) ---------------------------------------------------
    def _f(self, x, shape):
        x = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
        return x.reshape(shape)

    def _params(self, params, rows):
        """params=(refs, values): values as a [rows][len(refs)] float64 array."""
        if params is None:
            return None
        refs, values = params
        return refs, self._f(values, (rows, len(refs)))

    def calc_p2(self, dt, q0, q1, params=None):
        q0 = np.atleast_2d(np.asarray(q0, float))
        B = q0.shape[0]
        q0, q1 = self._f(q0, (B, self.nq)), self._f(q1, (B, self.nq))
        p = np.empty((B, self.nd))
        self.calc_p2_raw(False, B, float(dt), q0, q1, p, params=self._params(params, B))
        return p

    def calc_f(self, t1, t2, q1, q2, p1, u1=None, lambda1=None, params=None):
        """Residual of the DEL equation [B][nd+nc] (_MidpointVI._calc_f, midpointvi.c:533-575)."""
        q1 = np.atleast_2d(np.asarray(q1, float))
        B = q1.shape[0]
        q1, q2, p1 = self._f(q1, (B, self.nq)), self._f(q2, (B, self.nq)), self._f(p1, (B, self.nd))
        u1 = None if (u1 is None or self.nu == 0) else self._f(u1, (B, self.nu))
        lam = None if (lambda1 is None or self.nc == 0) else self._f(lambda1, (B, self.nc))
        f = np.empty((B, self.nd + self.nc))
        self.calc_f_raw(False, B, float(t1), float(t2), q1, q2, p1, u1, lam, f, params=self._params(params, B))
        return f

    def discrete_fm2(self, t1, t2, q1, q2, u1=None, params=None):
        """Discrete forcing (t2 - t1) F(q_mid, dq, u1) [B][nd] (_MidpointVI.discrete_fm2, midpointvi.c:2710-2727)."""
        q1 = np.atleast_2d(np.asarray(q1, float))
        B = q1.shape[0]
        q1, q2 = self._f(q1, (B, self.nq)), self._f(q2, (B, self.nq))
        u1 = None if (u1 is None or self.nu == 0) else self._f(u1, (B, self.nu))
        fm2 = np.empty((B, self.nd))
        self.discrete_fm2_raw(False, B, float(t1), float(t2), q1, q2, u1, fm2, params=self._params(params, B))
        return fm2

    def step(self, q1, p1, t0, dt, nsteps=1, u1=None, k2=None, q2_guess=None, lambda_guess=None,
             tolerance=1e-10, max_iterations=200, sample_every=0, times=None, params=None):
        """`nsteps` consecutive MidpointVI steps for every instance.  Returns a dict with the
        final q2, p2, lambda1, iters (summed), status and optionally the sampled trajectory.
        times: optional grid [nsteps+1] shared by the batch (step s runs times[s] -> times[s+1]).
        params: None, or (refs, values [B][len(refs)]): per-instance values of the SystemDesc.param_ref entries
        refs (the same keyword on linearize, project, calc_p2, calc_f and discrete_fm2)."""
        if times is not None:
            times = self._f(times, (nsteps + 1,))
        q1 = np.atleast_2d(np.asarray(q1, float))
        B = q1.shape[0]
        q1, p1 = self._f(q1, (B, self.nq)), self._f(p1, (B, self.nd))
        u1 = None if (u1 is None or self.nu == 0) else self._f(u1, (B, nsteps, self.nu))
        if self.nk:
            if k2 is None:
                raise ValueError("k2 [B][nsteps][nk] is required: the system has %d kinematic configs" % self.nk)
            k2 = self._f(k2, (B, nsteps, self.nk))
        else:
            k2 = None
        q2g = None if q2_guess is None else self._f(q2_guess, (B, self.nd))
        lg = None if (lambda_guess is None or self.nc == 0) else self._f(lambda_guess, (B, self.nc))
        out = dict(q2=np.empty((B, self.nq)), p2=np.empty((B, self.nd)),
                   lambda1=np.zeros((B, self.nc)), iters=np.zeros(B, np.int32),
                   status=np.zeros(B, np.int32))
        ns = nsteps // sample_every if sample_every > 0 else 0
        if ns:
            out["traj_q"] = np.empty((B, ns, self.nq))
            out["traj_p"] = np.empty((B, ns, self.nd))
        self.step_raw(False, B, nsteps, float(t0), float(dt), q1, p1, u1, k2, q2g, lg, out["q2"],
                      out["p2"], out["lambda1"] if self.nc else None, out["iters"], out["status"],
                      tolerance, max_iterations, sample_every, out.get("traj_q"), out.get("traj_p"), times=times,
                      params=self._params(params, B))
        return out

    def project(self, bX, bU, Kfb, t0, dt, use_hint=True, tolerance=1e-10, max_iterations=200, times=None, params=None):
        """Closed-loop rollouts X[0] = bX[0], U[k] = bU[k] - K[k](X[k] - bX[k]), X[k+1] = f(X[k], U[k])
        (DSystem.project / DOptimizer.armijo_simulate) for a batch of candidates.
        bX [B,K+1,nX], bU [B,K,nU], Kfb [K,nU,nX] (shared) or [B,K,nU,nX]."""
        bX = np.ascontiguousarray(np.asarray(bX, float))
        if bX.ndim == 2:
            bX = bX[None]
        B, K = bX.shape[0], bX.shape[1] - 1
        bX = self._f(bX, (B, K + 1, self.nX))
        bU = self._f(bU, (B, K, self.nU))
        Kfb = np.ascontiguousarray(np.asarray(Kfb, float))
        per = Kfb.ndim == 4
        Kfb = self._f(Kfb, (B, K, self.nU, self.nX) if per else (K, self.nU, self.nX))
        out = dict(X=np.zeros((B, K + 1, self.nX)), U=np.zeros((B, K, self.nU)), iters=np.zeros(B, np.int32),
                   status=np.zeros(B, np.int32), fail_step=np.zeros(B, np.int32))
        self.project_raw(False, B, K, float(t0), float(dt), bX, bU, Kfb, out["X"], out["U"], out["status"],
                         k_per_instance=per, use_hint=use_hint, iters=out["iters"], fail_step=out["fail_step"],
                         tolerance=tolerance, max_iterations=max_iterations,
                         times=None if times is None else self._f(times, (K + 1,)), params=self._params(params, B))
        return out

    def linearize(self, q1, p1, u1=None, k2=None, t1=0.0, t2=None, dt=None, q2_guess=None,
                  lambda_guess=None, want_raw=False, tolerance=1e-10, max_iterations=200, params=None):
        """One DSystem-style linearization per instance: solve the step, then A (fdx) and B (fdu).
        params: None, or (refs, values [B][len(refs)]) per-instance parameters."""
        q1 = np.atleast_2d(np.asarray(q1, float))
        B = q1.shape[0]
        q1, p1 = self._f(q1, (B, self.nq)), self._f(p1, (B, self.nd))
        u1 = self._f(u1 if u1 is not None else np.zeros((B, self.nu)), (B, self.nu))
        k2 = self._f(k2 if k2 is not None else np.zeros((B, self.nk)), (B, self.nk))
        q2g = None if q2_guess is None else self._f(q2_guess, (B, self.nd))
        lg = None if (lambda_guess is None or self.nc == 0) else self._f(lambda_guess, (B, self.nc))
        t1a = t2a = None
        t1s = dts = 0.0
        if np.ndim(t1) == 0 and (t2 is None or np.ndim(t2) == 0):
            t1s = float(t1)
            dts = float(dt) if t2 is None else float(t2) - float(t1)
            if t2 is not None:
                # keep the reference's dt = t2 - t1 rounding: pass both as arrays
                t1a = np.full(B, float(t1)); t2a = np.full(B, float(t2))
        else:
            t1a = self._f(np.broadcast_to(t1, (B,)), (B,))
            t2a = self._f(np.broadcast_to(t2, (B,)), (B,))
        out = dict(q2=np.empty((B, self.nq)), p2=np.empty((B, self.nd)), lambda1=np.zeros((B, self.nc)),
                   iters=np.zeros(B, np.int32), status=np.zeros(B, np.int32),
                   A=np.empty((B, self.nX, self.nX)), B=np.zeros((B, self.nX, self.nU)))
        rawbufs = {}
        if want_raw:
            wrt = {"dq1": self.nq, "dp1": self.nd, "du1": self.nu, "dk2": self.nk}
            for n in RAW:
                rawbufs[n] = np.zeros((B, wrt[n[3:]], self.nc if n.startswith("l1") else self.nd))
            out.update(rawbufs)
        self.linearize_raw(False, B, q1, p1, u1 if self.nu else None, k2 if self.nk else None,
                           out["status"], t1=t1a, t2=t2a, t1_scalar=t1s, dt_scalar=dts, q2_guess=q2g,
                           lambda_guess=lg, q2=out["q2"], p2=out["p2"],
                           lambda1=out["lambda1"] if self.nc else None, iters=out["iters"],
                           A=out["A"], B=out["B"] if self.nU else None,
                           raw={k: v for k, v in rawbufs.items() if v.size},
                           tolerance=tolerance, max_iterations=max_iterations, params=self._params(params, B))
        return out

    def d2_shapes(self, B):
        cnt = {"dq1": self.nq, "dp1": self.nd, "du1": self.nu, "dk2": self.nk}
        out = {}
        for w in D2_WHICH:
            for kd in D2_KINDS:
                a, b = kd[:3], kd[3:]
                out[w + "_" + kd] = (B, cnt[a], cnt[b], self.nc if w == "l1" else self.nd)
        return out

    def deriv2(self, q1, p1, u1=None, k2=None, t1=0.0, t2=None, dt=None, q2_guess=None,
               lambda_guess=None, tolerance=1e-10, max_iterations=200, z=None, tensors=True, params=None):
        """solve + first derivatives + every second-derivative tensor (reference layout
        [B][wrt A][wrt B][out]); returns the dict of `linearize(want_raw=True)` plus the tensors.
        params: None, or (refs, values [B][len(refs)]) per-instance parameters."""
        q1 = np.atleast_2d(np.asarray(q1, float))
        B = q1.shape[0]
        q1, p1 = self._f(q1, (B, self.nq)), self._f(p1, (B, self.nd))
        u1 = self._f(u1 if u1 is not None else np.zeros((B, self.nu)), (B, self.nu))
        k2 = self._f(k2 if k2 is not None else np.zeros((B, self.nk)), (B, self.nk))
        q2g = None if q2_guess is None else self._f(q2_guess, (B, self.nd))
        lg = None if (lambda_guess is None or self.nc == 0) else self._f(lambda_guess, (B, self.nc))
        t1a = self._f(np.broadcast_to(t1, (B,)), (B,))
        t2a = self._f(np.broadcast_to(t1a + dt if t2 is None else t2, (B,)), (B,))
        out = dict(q2=np.empty((B, self.nq)), p2=np.empty((B, self.nd)), lambda1=np.zeros((B, self.nc)),
                   iters=np.zeros(B, np.int32), status=np.zeros(B, np.int32),
                   A=np.empty((B, self.nX, self.nX)), B=np.zeros((B, self.nX, self.nU)))
        wrt = {"dq1": self.nq, "dp1": self.nd, "du1": self.nu, "dk2": self.nk}
        rawbufs = {n: np.zeros((B, wrt[n[3:]], self.nc if n.startswith("l1") else self.nd)) for n in RAW}
        d2 = {n: np.zeros(sh) for n, sh in self.d2_shapes(B).items()} if tensors else {}
        zk = {}
        if z is not None:
            zk = dict(z=self._f(z, (B, self.nX)), fdxdx=np.zeros((B, self.nX, self.nX)),
                      fdxdu=np.zeros((B, self.nX, self.nU)), fdudu=np.zeros((B, self.nU, self.nU)))
            out.update({k: v for k, v in zk.items() if k != "z"})
            if not self.nU:
                zk["fdxdu"] = zk["fdudu"] = None
        self.deriv2_raw(False, B, q1, p1, u1 if self.nu else None, k2 if self.nk else None, out["status"],
                        {n: v for n, v in d2.items() if v.size}, **zk, t1=t1a, t2=t2a, q2_guess=q2g,
                        lambda_guess=lg, q2=out["q2"], p2=out["p2"],
                        lambda1=out["lambda1"] if self.nc else None, iters=out["iters"], A=out["A"],
                        B=out["B"] if self.nU else None, raw={k: v for k, v in rawbufs.items() if v.size},
                        tolerance=tolerance, max_iterations=max_iterations, params=self._params(params, B))
        out.update(rawbufs)
        out.update(d2)
        return out
