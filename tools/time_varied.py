"""Per-instance physical parameters (trepb_*_varied_batch_dev) against the plain entry points on the same handle, same
inputs, alternating in one process; CUDA events around each call (the varied calls' map upload included).

  W2 shape:  2^20 damped pendulums x 1000 steps, each with its own mass, length and damping coefficient
  W3 shape:  pend-on-cart linearize along 4096 trajectories of 10k steps (exact hints), one parameter set per trajectory
  single:    pend-on-cart single-step linearize of 2^22 random states, one parameter set per instance
  table:     fourbar on the table-driven thread kernels (TREPB_FLAG_NO_SPECIALIZE), 2^18 instances: 100 steps, and
             one linearize

Usage: python tools/time_varied.py [--reps 5] [--small]     (--small: 1/64 of every size, a quick rehearsal)
Prints one JSON line per workload: plain and varied ms (median of reps), their ratio, the card and its power limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from trep_b200 import lib, systems  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception:
        return "unknown", "unknown"


class At:
    """A device address inside another buffer."""
    def __init__(self, p):
        self.p = p

    def data_ptr(self):
        return self.p


def up(a):
    a = np.ascontiguousarray(a)
    return lib.DeviceBuffer(0, a.shape, a.dtype).upload(a)


def timed(fn, reps):
    fn(False), fn(True)                     # warm-up: module load, scratch, map upload path
    t = {False: [], True: []}
    for _ in range(reps):
        for varied in (False, True):
            with lib.EventTimer(0) as ev:
                fn(varied)
            t[varied].append(ev.ms)
    return float(np.median(t[False])), float(np.median(t[True]))


def report(name, plain, varied, extra, gpu):
    print(json.dumps(dict(workload=name, plain_ms=round(plain, 3), varied_ms=round(varied, 3),
                          ratio=round(varied / plain, 4), card=gpu[0], power_limit=gpu[1], **extra)), flush=True)


def params(d, refs, rows, rng, spread=0.5):
    base = np.array([d.param_value(r) for r in refs])
    return base * rng.uniform(1 - spread, 1 + spread, (rows, len(refs)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--small", action="store_true")
    a = ap.parse_args()
    f = 64 if a.small else 1
    gpu = card()
    rng = np.random.default_rng(0)

    # W2 shape
    d = systems.named_desc("damped_pendulum")
    s = lib.System(d)
    refs = [d.param_ref("frame_mass", 3, 0), d.param_ref("frame_value", 3), d.param_ref("dpool", 0)]
    B, K = (1 << 20) // f, 1000
    q1, p1 = up(rng.uniform(-1, 1, (B, 1))), up(np.zeros((B, 1)))
    q2, p2 = lib.DeviceBuffer(0, (B, 1)), lib.DeviceBuffer(0, (B, 1))
    it, st = lib.DeviceBuffer(0, (B,), np.int32), lib.DeviceBuffer(0, (B,), np.int32)
    dv = up(params(d, refs, B, rng))
    run = lambda v: s.step_raw(True, B, K, 0.0, 0.01, q1, p1, None, None, None, None, q2, p2, None, it, st,
                               params=(refs, dv) if v else None)
    pl, va = timed(run, a.reps)
    report("W2_step_damped_pendulum", pl, va, dict(batch=B, nsteps=K, varied=len(refs), kernel=s.kernel_name,
                                                    steps_per_s_plain=B * K / pl * 1e3, steps_per_s_varied=B * K / va * 1e3), gpu)
    del q1, p1, q2, p2, it, st, dv

    # W3 shape: linearize along trajectories, one row per trajectory
    d = systems.named_desc("pend_on_cart1")
    s = lib.System(d)
    refs = [d.param_ref("frame_mass", 3, 0), d.param_ref("frame_value", 3), d.param_ref("dpool", 0), d.param_ref("dpool", 1)]
    refs = [r for r in refs if d.param_value(r) != 0.0]
    R, L = 4096 // f, 10000
    q0 = rng.uniform(-0.5, 0.5, (R, d.nq)); p0 = np.zeros((R, d.nd))
    u = rng.uniform(-0.5, 0.5, (R, L - 1, d.nu))
    tr = s.step(q0, p0, 0.0, 0.01, nsteps=L - 1, u1=u, sample_every=1)
    X = np.concatenate([q0[:, None], tr["traj_q"]], 1)
    P = np.concatenate([p0[:, None], tr["traj_p"]], 1)
    n = R * (L - 1)
    dq, dp, du = up(X), up(P), up(u)
    hint = At(dq.ptr + 8 * d.nq)            # X[k+1] as the Newton start (trepb_lin_args.traj_len)
    A = lib.DeviceBuffer(0, (n, d.nX, d.nX)); Bm = lib.DeviceBuffer(0, (n, d.nX, d.nU))
    st = lib.DeviceBuffer(0, (n,), np.int32)
    dv = up(params(d, refs, R, rng, 0.0))   # the trajectories were made with the base numbers: exact hints
    run = lambda v: s.linearize_raw(True, n, dq, dp, du, None, st, t1_scalar=0.0, dt_scalar=0.01, q2_guess=hint,
                                    A=A, B=Bm, traj_len=L, params=(refs, dv) if v else None)
    pl, va = timed(run, a.reps)
    report("W3_linearize_trajectories_pend_on_cart1", pl, va, dict(trajectories=R, traj_len=L, varied=len(refs),
                                                                   kernel=s.kernel_name, lin_per_s_plain=n / pl * 1e3,
                                                                   lin_per_s_varied=n / va * 1e3), gpu)
    del dq, dp, du, A, Bm, st, dv

    # single-step linearize, one set per instance
    B = (1 << 22) // f
    dq, dp = up(rng.uniform(-1, 1, (B, d.nq))), up(rng.normal(0, 0.5, (B, d.nd)))
    du = up(rng.uniform(-0.5, 0.5, (B, d.nu)))
    A = lib.DeviceBuffer(0, (B, d.nX, d.nX)); Bm = lib.DeviceBuffer(0, (B, d.nX, d.nU))
    st = lib.DeviceBuffer(0, (B,), np.int32)
    dv = up(params(d, refs, B, rng))
    run = lambda v: s.linearize_raw(True, B, dq, dp, du, None, st, t1_scalar=0.0, dt_scalar=0.01, A=A, B=Bm,
                                    params=(refs, dv) if v else None)
    pl, va = timed(run, a.reps)
    report("single_step_linearize_pend_on_cart1", pl, va, dict(batch=B, varied=len(refs), kernel=s.kernel_name,
                                                               lin_per_s_plain=B / pl * 1e3, lin_per_s_varied=B / va * 1e3), gpu)
    del dq, dp, du, A, Bm, st, dv

    # table-driven thread kernels
    d = systems.named_desc("fourbar")
    s = lib.System(d, specialize=False, cooperative=False)
    g = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "fourbar.npz"))
    B = (1 << 18) // f
    idx = np.arange(B) % len(g["case_iters"])
    refs = [d.param_ref("frame_mass", f_, 0) for f_ in range(d.n_frames) if d.frame_mass[f_, 0] != 0.0]
    refs += [(6, i) for i in range(len(d.dpool)) if d.dpool[i] != 0.0]
    dq, dp = up(g["case_q1"][idx]), up(g["case_p1"][idx])
    du = up(g["case_u1"][idx]) if d.nu else None
    dk = up(np.repeat(g["case_k2"][idx][:, None], 100, 1)) if d.nk else None
    q2, p2 = lib.DeviceBuffer(0, (B, d.nq)), lib.DeviceBuffer(0, (B, d.nd))
    lam = lib.DeviceBuffer(0, (B, max(d.nc, 1)))
    it, st = lib.DeviceBuffer(0, (B,), np.int32), lib.DeviceBuffer(0, (B,), np.int32)
    dv = up(params(d, refs, B, rng, 0.2))
    du100 = up(np.repeat(g["case_u1"][idx][:, None], 100, 1)) if d.nu else None
    run = lambda v: s.step_raw(True, B, 100, 0.0, 0.01, dq, dp, du100, dk, None, None, q2, p2, lam if d.nc else None,
                               it, st, params=(refs, dv) if v else None)
    pl, va = timed(run, a.reps)
    report("table_driven_step_fourbar", pl, va, dict(batch=B, nsteps=100, varied=len(refs), kernel=s.kernel_name), gpu)
    A = lib.DeviceBuffer(0, (B, d.nX, d.nX))
    dk1 = up(g["case_k2"][idx]) if d.nk else None
    run = lambda v: s.linearize_raw(True, B, dq, dp, du, dk1, st, t1_scalar=0.0, dt_scalar=0.01, A=A,
                                    params=(refs, dv) if v else None)
    pl, va = timed(run, a.reps)
    report("table_driven_linearize_fourbar", pl, va, dict(batch=B, varied=len(refs), kernel=s.kernel_name), gpu)


if __name__ == "__main__":
    main()
