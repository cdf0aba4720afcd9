"""Per-instance physical parameters on the cooperative kernels (TREPB_FLAG_COOP_VARIED), timed three ways on the same
inputs, alternating in one process, CUDA events around each call (median of reps):
  varied     varied call on a flagged cooperative handle (the varied cooperative kernels)
  plain      plain call on the same handle (every instance on the description's numbers)
  no_coop    varied call on a TREPB_FLAG_NO_COOP handle (the table-driven thread kernels, the only way before)

Workloads, on the marionette unless named otherwise:
  lin_traj_<R>    linearize along R trajectories x 1000 steps, one row per trajectory (R = 148, 1184; A written for
                  148 only: 1184 x 999 A matrices would take 60 GB)
  lin_single      single-step linearize of 2^16 instances, one row each
  step / project  1184 rollouts x 1000 steps, one row each
  deriv2          1024 instances, z-contracted
  doptimizer      one DOptimizer.step (newton), 16 rollouts x 100 steps, with per-rollout rows against the same
                  step without rows (host clock around the call, which ends in a device synchronise)
  pccd_lin_traj   pccd linearize along 148 trajectories x 1000 steps

Usage: python tools/time_varied_coop.py [--reps 3] [--small]     (--small: 1/8 of the batch sizes, a quick rehearsal)
Prints one JSON line per workload with the card and its power limit, read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from time_varied import At, card, up  # noqa: E402
from trep_b200 import lib, systems  # noqa: E402


def refs_of(d):
    """Every entry that may vary, without the frame_se3 ones (a row keeps the rotations orthonormal)."""
    out = []
    for t, name in enumerate(("frame_value", "frame_se3", "frame_mass", "pot_d", "force_d", "con_d", "dpool")):
        if name == "frame_se3":
            continue
        for i, v in enumerate(getattr(d, name).reshape(-1)):
            if v != 0.0:
                out.append((t, i))
    try:
        lib.check_params(d, out)
    except lib.TrepbError:
        from test_varied_params import variable_refs
        out = [r for r in variable_refs(d) if r[0] != 1]
    return out


def rows(d, refs, n, rng, spread=0.02):
    base = np.array([d.param_value(r) for r in refs])
    return base * rng.uniform(1 - spread, 1 + spread, (n, len(refs)))


def timed(fns, reps):
    for f in fns.values():
        f()                                  # warm-up: module load, scratch, plan upload
    t = {k: [] for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            with lib.EventTimer(0) as ev:
                f()
            t[k].append(ev.ms)
    return {k: float(np.median(v)) for k, v in t.items()}


def report(name, t, extra, gpu):
    out = dict(workload=name, **{k + "_ms": round(v, 3) for k, v in t.items()})
    if "plain" in t:
        out["varied_over_plain"] = round(t["varied"] / t["plain"], 4)
    if "no_coop" in t:
        out["no_coop_over_varied"] = round(t["no_coop"] / t["varied"], 4)
    out.update(card=gpu[0], power_limit=gpu[1], **extra)
    print(json.dumps(out), flush=True)


def golden(name):
    return np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))


def trajectories(s, d, g, R, L, rng):
    idx = np.arange(R) % len(g["case_iters"])
    q0, p0 = g["case_q1"][idx], g["case_p1"][idx]
    u = np.repeat(g["case_u1"][idx][:, None], L - 1, 1) if d.nu else None
    k = (g["case_k2"][idx][:, None] + 1e-4 * np.arange(1, L)[None, :, None]) if d.nk else None
    tr = s.step(q0, p0, 0.0, 0.01, nsteps=L - 1, u1=u, k2=k, sample_every=1)
    X = np.concatenate([q0[:, None], tr["traj_q"]], 1)
    P = np.concatenate([p0[:, None], tr["traj_p"]], 1)
    return X, P, u, k


def lin_traj(name, d, g, handles, R, L, with_A, rng, gpu):
    s, nc = handles
    refs = refs_of(d)
    X, P, u, k = trajectories(s, d, g, R, L, rng)
    n = R * (L - 1)
    dq, dp = up(X), up(P)
    du = up(u) if d.nu else None
    dk = up(k) if d.nk else None
    hint = At(dq.ptr + 8 * d.nq)
    A = lib.DeviceBuffer(0, (n, d.nX, d.nX)) if with_A else None
    st = lib.DeviceBuffer(0, (n,), np.int32)
    dv = up(rows(d, refs, R, rng))
    run = lambda h, v: (lambda: h.linearize_raw(True, n, dq, dp, du, dk, st, t1_scalar=0.0, dt_scalar=0.01,
                                                q2_guess=hint, A=A, traj_len=L, params=(refs, dv) if v else None))
    t = timed(dict(varied=run(s, True), plain=run(s, False), no_coop=run(nc, True)), REPS)
    report(name, t, dict(trajectories=R, traj_len=L, A=with_A, kernel=s.kernel_name,
                         lin_per_s_varied=n / t["varied"] * 1e3, lin_per_s_plain=n / t["plain"] * 1e3,
                         lin_per_s_no_coop=n / t["no_coop"] * 1e3), gpu)


def main():
    global REPS
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--small", action="store_true")
    a = ap.parse_args()
    REPS = a.reps
    f = 8 if a.small else 1
    gpu = card()
    rng = np.random.default_rng(0)
    d, g = systems.named_desc("puppet"), golden("puppet")
    refs = refs_of(d)
    s = lib.System(d, coop_varied=True)
    nc = lib.System(d, cooperative=False)
    assert s.cooperative and not nc.cooperative

    lin_traj("lin_traj_148", d, g, (s, nc), max(148 // f, 2), 1000, True, rng, gpu)
    lin_traj("lin_traj_1184", d, g, (s, nc), 1184 // f, 1000, False, rng, gpu)

    # single-step linearize, one row per instance
    B = (1 << 16) // f
    idx = np.arange(B) % len(g["case_iters"])
    dq, dp, dk = up(g["case_q1"][idx]), up(g["case_p1"][idx]), up(g["case_k2"][idx])
    du = up(g["case_u1"][idx]) if d.nu else None
    A = lib.DeviceBuffer(0, (B, d.nX, d.nX))
    st = lib.DeviceBuffer(0, (B,), np.int32)
    dv = up(rows(d, refs, B, rng))
    run = lambda h, v: (lambda: h.linearize_raw(True, B, dq, dp, du, dk, st, t1_scalar=0.0, dt_scalar=0.01, A=A,
                                                params=(refs, dv) if v else None))
    t = timed(dict(varied=run(s, True), plain=run(s, False), no_coop=run(nc, True)), REPS)
    report("lin_single", t, dict(batch=B, kernel=s.kernel_name, lin_per_s_varied=B / t["varied"] * 1e3), gpu)
    del A

    # step and project: 1184 rollouts x 1000 steps
    B, K = 1184 // f, 1000
    idx = np.arange(B) % len(g["case_iters"])
    dq, dp = up(g["case_q1"][idx]), up(g["case_p1"][idx])
    dk = up(g["case_k2"][idx][:, None] + 1e-4 * np.arange(1, K + 1)[None, :, None])
    du = up(np.repeat(g["case_u1"][idx][:, None], K, 1)) if d.nu else None
    q2, p2 = lib.DeviceBuffer(0, (B, d.nq)), lib.DeviceBuffer(0, (B, d.nd))
    lam = lib.DeviceBuffer(0, (B, d.nc))
    it, st = lib.DeviceBuffer(0, (B,), np.int32), lib.DeviceBuffer(0, (B,), np.int32)
    dv = up(rows(d, refs, B, rng))
    run = lambda h, v: (lambda: h.step_raw(True, B, K, 0.0, 0.01, dq, dp, du, dk, None, None, q2, p2, lam, it, st,
                                           params=(refs, dv) if v else None))
    t = timed(dict(varied=run(s, True), plain=run(s, False), no_coop=run(nc, True)), REPS)
    report("step", t, dict(rollouts=B, nsteps=K, steps_per_s_varied=B * K / t["varied"] * 1e3), gpu)
    bXh = np.zeros((B, K + 1, d.nX))
    bXh[:, :, :d.nq] = g["case_q1"][idx][:, None]
    bXh[:, :, d.nq:d.nq + d.nd] = g["case_p1"][idx][:, None]
    bUh = np.zeros((B, K, d.nU))
    bUh[:, :, d.nu:] = g["case_k2"][idx][:, None] + 1e-4 * np.arange(1, K + 1)[None, :, None]
    bX, bU = up(bXh), up(bUh)
    Kfb = up(rng.normal(0, 0.01, (K, d.nU, d.nX)))
    X, U = lib.DeviceBuffer(0, (B, K + 1, d.nX)), lib.DeviceBuffer(0, (B, K, d.nU))
    run = lambda h, v: (lambda: h.project_raw(True, B, K, 0.0, 0.01, bX, bU, Kfb, X, U, st, iters=it,
                                              params=(refs, dv) if v else None))
    t = timed(dict(varied=run(s, True), plain=run(s, False), no_coop=run(nc, True)), REPS)
    report("project", t, dict(rollouts=B, nsteps=K, steps_per_s_varied=B * K / t["varied"] * 1e3), gpu)
    del bX, bU, X, U, dk

    # second derivatives, z-contracted
    B = 1024 // f
    idx = np.arange(B) % len(g["case_iters"])
    z = rng.normal(0, 1, (B, d.nX))
    P = (refs, rows(d, refs, B, rng))
    kw = dict(t1=0.0, t2=0.01, z=z, tensors=False)
    args = (g["case_q1"][idx], g["case_p1"][idx], g["case_u1"][idx] if d.nu else None, g["case_k2"][idx])
    t = timed(dict(varied=lambda: s.deriv2(*args, params=P, **kw), plain=lambda: s.deriv2(*args, **kw),
                   no_coop=lambda: nc.deriv2(*args, params=P, **kw)), REPS)
    report("deriv2_z", t, dict(batch=B, note="host-pointer calls: staging included"), gpu)

    # DOptimizer.step (newton), 16 x 100, per-rollout rows against none
    from trep_b200 import discopt, midpointvi as MV
    R, K = 16, 100
    tt = np.arange(K + 1) * 0.01
    idx = np.arange(R) % len(g["case_iters"])
    ds = discopt.DSystem(MV.MidpointVI(d), tt)
    Xh = np.zeros((R, K + 1, d.nX))
    Xh[:, :, :d.nq] = g["case_q1"][idx][:, None]
    Xh[:, :, d.nq:d.nq + d.nd] = g["case_p1"][idx][:, None]
    Uh = np.zeros((R, K, d.nU))
    Uh[:, :, d.nu:] = g["case_k2"][idx][:, None] + 1e-4 * np.arange(1, K + 1)[None, :, None]
    Xh = ds.simulate(Xh[:, 0], Uh)
    cost = discopt.DCost(Xh + 0.01, Uh, np.eye(d.nX), 0.1 * np.eye(d.nU))
    vals = rows(d, refs, R, rng)
    times = {"varied": [], "plain": []}
    for rep in range(REPS + 1):
        for mode in ("varied", "plain"):
            ds.set_parameters(*((refs, vals) if mode == "varied" else (None, None)))
            opt = discopt.DOptimizer(ds, cost)
            t0 = time.perf_counter()
            opt.step(0, Xh, Uh, "newton")
            if rep:
                times[mode].append((time.perf_counter() - t0) * 1e3)
    report("doptimizer_newton", {k: float(np.median(v)) for k, v in times.items()},
           dict(rollouts=R, nsteps=K, clock="host"), gpu)

    # pccd
    d, g = systems.named_desc("pccd"), golden("pccd")
    sp, ncp = lib.System(d, coop_varied=True), lib.System(d, cooperative=False)
    assert sp.cooperative
    lin_traj("pccd_lin_traj_148", d, g, (sp, ncp), max(148 // f, 2), 1000, True, rng, gpu)


if __name__ == "__main__":
    main()
