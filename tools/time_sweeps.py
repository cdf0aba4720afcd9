"""Tangent and adjoint sweeps (trepb_tangent_batch_dev, trepb_adjoint_batch_dev): kernel time and HBM fraction, the
host path they replace, and DSystem.calc_descent_direction end to end against the calls it replaces.

  kernel:      CUDA events around each _dev call, median of `reps` alternating (tangent, adjoint) pairs after one
               warm-up each.  Bytes = R K 8 (nX^2 + 2 nX nU) (A, B and K once each; the vectors are not counted),
               fraction over 7.7 TB/s.  Inputs are drawn on the device (torch), A scaled to spectral radius ~0.9.
  host path:   download of A / B / K (torch .cpu()) plus the numpy recursion of DSystem.dproject / the costate loop of
               DSystem.calc_newton_model on the same inputs (shapes whose slabs fit in host memory only).
  end to end:  DSystem.calc_descent_direction(newton=False / True) against calc_feedback_controller(
               return_linearization=True) [+ calc_newton_model] + lib.solve_tv_lq + the host loop, host clock around
               each (both synchronize), median of 3 alternating.

Usage: python tools/time_sweeps.py [--reps 5] [--skip-host] [--skip-e2e]
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

# (label, rollouts, steps, nX, nU, host path measured)
KERNEL_SHAPES = [("pend-on-cart W3", 4096, 10000, 4, 1, True),
                 ("marionette dims", 148, 1000, 80, 18, True),
                 ("marionette dims", 1184, 1000, 80, 18, False),
                 ("pend-on-cart, one rollout", 1, 10000, 4, 1, True),
                 ("marionette dims, one rollout", 1, 10000, 80, 18, True)]


def emit(gpu, **row):
    print(json.dumps(dict(row, card=gpu[0], power_limit=gpu[1])), flush=True)


def kernels(gpu, reps, host):
    import torch
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)
    for label, R, K, nX, nU, host_ok in KERNEL_SHAPES:
        rnd = lambda *s, sc=1.0: torch.randn(*s, device=dev, dtype=torch.float64, generator=g).mul_(sc)
        A = rnd(R, K, nX, nX, sc=0.9 / np.sqrt(nX))
        B = rnd(R, K, nX, nU, sc=0.3 / np.sqrt(nX))
        Kf = rnd(R, K, nU, nX, sc=0.1 / np.sqrt(nX))
        bdU, m_dx, l_dx = rnd(R, K, nU), rnd(R, nX), rnd(R, K, nX)
        dX, dU = torch.empty(R, K + 1, nX, device=dev, dtype=torch.float64), torch.empty(R, K, nU, device=dev, dtype=torch.float64)
        z = torch.empty(R, K + 1, nX, device=dev, dtype=torch.float64)
        torch.cuda.synchronize()
        tangent = lambda: lib.tangent_raw(True, 0, R, K, nX, nU, A, B, Kf, dX, dU, bdU=bdU)
        adjoint = lambda: lib.adjoint_raw(True, 0, R, K, nX, nU, A, B, m_dx, z, K=Kf, l_dx=l_dx, l_du=bdU)
        tangent(), adjoint()
        t = {"tangent": [], "adjoint": []}
        for _ in range(reps):
            for name, fn in (("tangent", tangent), ("adjoint", adjoint)):
                with lib.EventTimer(0) as ev:
                    fn()
                t[name].append(ev.ms)
        nbytes = R * K * 8 * (nX * nX + 2 * nX * nU)
        row = dict(table="kernel", shape=label, rollouts=R, steps=K, nX=nX, nU=nU, gbytes=round(nbytes / 1e9, 3))
        for name in t:
            ms = float(np.median(t[name]))
            row[name + "_ms"] = round(ms, 3)
            row[name + "_hbm_fraction"] = round(nbytes / (ms * 1e-3) / HBM, 3)
        if host and host_ok:
            t0 = time.perf_counter()
            hA, hB, hK, hbdU = A.cpu().numpy(), B.cpu().numpy(), Kf.cpu().numpy(), bdU.cpu().numpy()
            hl, hm = l_dx.cpu().numpy(), m_dx.cpu().numpy()
            t1 = time.perf_counter()
            bdX = np.zeros((R, K + 1, nX))
            want = discopt.DSystem.dproject(discopt.DSystem, hA, hB, bdX, hbdU, hK)
            t2 = time.perf_counter()
            Z = np.zeros((R, K + 1, nX)); Z[:, K] = hm
            for k in reversed(range(K)):
                Acl = hA[:, k] - np.einsum("rxu,ruy->rxy", hB[:, k], hK[:, k])
                Z[:, k] = hl[:, k] - np.einsum("ru,rux->rx", hbdU[:, k], hK[:, k]) + np.einsum("rx,rxy->ry", Z[:, k + 1], Acl)
            t3 = time.perf_counter()
            row.update(host_download_ms=round(1e3 * (t1 - t0), 1), host_dproject_ms=round(1e3 * (t2 - t1), 1),
                       host_costate_ms=round(1e3 * (t3 - t2), 1))
            # the device results on the same inputs, for the record
            row["tangent_max_rel_diff"] = float(np.max(np.abs(dX.cpu().numpy() - want.dX)) / max(np.max(np.abs(want.dX)), 1e-300))
            row["adjoint_max_rel_diff"] = float(np.max(np.abs(z.cpu().numpy() - Z)) / max(np.max(np.abs(Z)), 1e-300))
            del hA, hB, hK, want, Z
        else:
            row.update(host_download_ms="not measured", host_dproject_ms="not measured", host_costate_ms="not measured")
        emit(gpu, **row)
        del A, B, Kf, bdU, m_dx, l_dx, dX, dU, z
        torch.cuda.empty_cache()


def end_to_end(gpu):
    import golden_util as G
    from test_gpu_sweeps import _composed, _dsys, _model
    from test_gpu_varied_deriv2 import _traj
    for name, R, K in (("pend_on_cart1", 64, 1000), ("puppet", 16, 100)):
        d, g = G.desc(name), G.golden(name)
        rng = np.random.default_rng(1)
        X, U = _traj(d, g, R, K, rng)
        ds = _dsys(d, np.arange(K + 1) * 0.01)
        q, r, Q, S, Rc = _model(ds, X, U, 2)
        for newton in (False, True):
            new = lambda: ds.calc_descent_direction(X, U, q, r, Q, S, Rc, newton=newton)
            old = lambda: _composed(ds, X, U, q, r, Q, S, Rc, newton)
            new(), old()
            t = {"new": [], "old": []}
            for _ in range(3):
                for k, fn in (("new", new), ("old", old)):
                    t0 = time.perf_counter()
                    fn()
                    t[k].append(1e3 * (time.perf_counter() - t0))
            a, b = float(np.median(t["new"])), float(np.median(t["old"]))
            emit(gpu, table="end_to_end", system=name, rollouts=R, steps=K, newton=newton,
                 calc_descent_direction_ms=round(a, 1), composed_ms=round(b, 1), speedup=round(b / a, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-host", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    a = ap.parse_args()
    if lib.device_count() < 1:
        raise SystemExit("time_sweeps.py needs a CUDA device")
    gpu = card()
    kernels(gpu, a.reps, not a.skip_host)
    if not a.skip_e2e:
        end_to_end(gpu)


if __name__ == "__main__":
    main()
