"""discopt.DOptimizer: the track kernel alone (trepb_track_batch_dev) and one optimiser step against the host
composition it replaces.

  kernel:  CUDA events around each _dev call, median of `reps` after one warm-up.  Two launches per shape: "gradient"
           (cost, q, r, l_dx, m_dx from X, U and one shared reference) and "newton model" (Qm, Sm, Rm from Q, R and
           the three Newton blocks).  Bytes are what each launch must move: gradient 8 R ((K+1) nX + K nU) x 2 read
           (trajectory and its reference) + 8 R ((K+1) nX + K nU + K nX + nX + 1) written; newton model
           8 R K (nX^2 + nX nU + nU^2) read + 8 R ((K+1) nX^2 + K nX nU + K nU^2) written.  Fraction over 7.7 TB/s.
           Inputs are drawn on the device (torch).
  step:    DOptimizer.step(method) against the host composition of tests/test_gpu_doptimizer.py (DSystem.
           calc_descent_direction with numpy model arrays, numpy DCost loops for cost / dcost, and the reference's
           one-candidate-at-a-time Armijo loop over DSystem.project), host clock around each, median of `step_reps`
           alternating; the accepted m of both is checked to agree.

Usage: python tools/time_doptimizer.py [--reps 20] [--step-reps 2] [--skip-step]
Prints one JSON line per row, each with the card and its power limit."""
import argparse
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
sys.path.insert(0, HERE)
from time_varied import card  # noqa: E402
from trep_b200 import discopt, lib  # noqa: E402

HBM = 7.7e12

# (label, trajectories, steps, nX, nU)
KERNEL_SHAPES = [("marionette dims", 16, 100, 80, 18),
                 ("marionette dims", 148, 1000, 80, 18),
                 ("pend-on-cart dims", 64, 1000, 4, 1),
                 ("pend-on-cart dims", 4096, 1000, 4, 1)]


def emit(gpu, **row):
    print(json.dumps(dict(row, card=gpu[0], power_limit=gpu[1])), flush=True)


def kernels(gpu, reps):
    import torch
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)
    for label, R, K, nX, nU in KERNEL_SHAPES:
        rnd = lambda *s: torch.randn(*s, device=dev, dtype=torch.float64, generator=g)
        emp = lambda *s: torch.empty(*s, device=dev, dtype=torch.float64)
        X, U, Xd, Ud = rnd(R, K + 1, nX), rnd(R, K, nU), rnd(1, K + 1, nX), rnd(1, K, nU)
        Q, Rw = torch.eye(nX, device=dev, dtype=torch.float64), torch.eye(nU, device=dev, dtype=torch.float64)
        q, r, l_dx, m_dx, cost = emp(R, K + 1, nX), emp(R, K, nU), emp(R, K, nX), emp(R, nX), emp(R)
        fxx, fxu, fuu = rnd(R * K, nX, nX), rnd(R * K, nX, nU), rnd(R * K, nU, nU)
        Qm, Sm, Rm = emp(R, K + 1, nX, nX), emp(R, K, nX, nU), emp(R, K, nU, nU)
        torch.cuda.synchronize()
        launches = {
            "gradient": (lambda: lib.track_raw(True, 0, R, K, nX, nU, X=X, U=U, Xd=Xd, Ud=Ud, Q=Q, R=Rw, q=q, r=r,
                                               l_dx=l_dx, m_dx=m_dx, cost=cost),
                         8 * R * (2 * ((K + 1) * nX + K * nU) + (K + 1) * nX + K * nU + K * nX + nX + 1)),
            "newton_model": (lambda: lib.track_raw(True, 0, R, K, nX, nU, Q=Q, R=Rw, fdxdx=fxx, fdxdu=fxu, fdudu=fuu,
                                                   Qm=Qm, Sm=Sm, Rm=Rm),
                             8 * R * (K * (nX * nX + nX * nU + nU * nU) + (K + 1) * nX * nX + K * nX * nU + K * nU * nU)),
        }
        for name, (fn, nbytes) in launches.items():
            fn()
            t = []
            for _ in range(reps):
                with lib.EventTimer(0) as ev:
                    fn()
                t.append(ev.ms)
            ms = float(np.median(t))
            emit(gpu, table="kernel", launch=name, shape=label, trajectories=R, steps=K, nX=nX, nU=nU,
                 gbytes=round(nbytes / 1e9, 4), ms=round(ms, 4), hbm_fraction=round(nbytes / (ms * 1e-3) / HBM, 3))
        del X, U, Xd, Ud, q, r, l_dx, m_dx, cost, fxx, fxu, fuu, Qm, Sm, Rm
        torch.cuda.empty_cache()


def steps(gpu, reps):
    from test_gpu_doptimizer import _problem, host_step
    for name, R, K in (("pend_on_cart1", 64, 1000), ("puppet", 16, 100)):
        d, t, ds, X, U, cost = _problem(name, R, K, 1)
        opt = discopt.DOptimizer(ds, cost)
        for method in ("newton", "quasi"):
            new = lambda: opt.step(0, X, U, method)
            old = lambda: host_step(opt, X, U, method)
            new()
            m_new = opt.last_armijo_m.copy()
            m_old = old()[-1]
            tm = {"new": [], "old": []}
            for _ in range(reps):
                for k, fn in (("new", new), ("old", old)):
                    t0 = time.perf_counter()
                    fn()
                    tm[k].append(1e3 * (time.perf_counter() - t0))
            a, b = float(np.median(tm["new"])), float(np.median(tm["old"]))
            emit(gpu, table="step", system=name, rollouts=R, steps=K, method=method, doptimizer_step_ms=round(a, 1),
                 host_composition_ms=round(b, 1), speedup=round(b / a, 2), same_accepted_m=bool(np.array_equal(m_new, m_old)),
                 accepted_m=[int(m) for m in m_new])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--step-reps", type=int, default=2)
    ap.add_argument("--skip-step", action="store_true")
    a = ap.parse_args()
    if lib.device_count() < 1:
        raise SystemExit("time_doptimizer.py needs a CUDA device")
    gpu = card()
    kernels(gpu, a.reps)
    if not a.skip_step:
        steps(gpu, a.step_reps)


if __name__ == "__main__":
    main()
