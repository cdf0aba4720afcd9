"""Stationary LQR: the DARE solve on the device (trepb_dare_batch_dev) against the host path it replaces.

  device:      CUDA events around the _dev call (inputs already in HBM), median of `reps` after one warm-up, at the
               pend-on-cart's dims (4 x 1) and the marionette's (80 x 18), for 1, 148 and 4096 models.  The models are
               random stabilizable problems (tests/test_gpu_dare.py's generator); the doubling steps taken are
               reported with the time.
  host:        what a user does without it: download A / B from the device, then scipy.linalg.solve_discrete_are
               and one solve for K per model (host clock, one pass; 4096 models at 80 x 18 are timed on 148 and
               scaled).
  end to end:  DSystem.calc_stationary_controller on pend-on-cart at the upright equilibrium under 148 models
               (set_parameters): upload, linearize, DARE, synchronize, download K and P (host clock, median of reps),
               against the same linearization followed by the host path.

Usage: python tools/time_dare.py [--reps 20]
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
from trep_b200 import discopt, lib, midpointvi as MV  # noqa: E402

SHAPES = [(4, 1), (80, 18)]
MODELS = [1, 148, 4096]


def emit(gpu, **row):
    print(json.dumps(dict(row, card=gpu[0], power_limit=gpu[1])), flush=True)


def host_dare(A, B, Q, R):
    import scipy.linalg as sla
    K = np.empty((A.shape[0], B.shape[2], A.shape[1]))
    for i in range(A.shape[0]):
        P = sla.solve_discrete_are(A[i], B[i], Q, R)
        K[i] = np.linalg.solve(R + B[i].T @ P @ B[i], B[i].T @ P @ A[i])
    return K


def device_rows(gpu, reps):
    import torch
    from test_gpu_dare import problem
    for nX, nU in SHAPES:
        for N in MODELS:
            A, B, Q, R, _ = problem(np.random.default_rng(N + nX), N, nX, nU)
            t = lambda x: torch.tensor(np.ascontiguousarray(x), device="cuda")
            dA, dB, dQ, dR = t(A), t(B), t(Q), t(R)
            dK = torch.empty((N, nU, nX), dtype=torch.float64, device="cuda")
            dP = torch.empty((N, nX, nX), dtype=torch.float64, device="cuda")
            dst, dit = (torch.empty(N, dtype=torch.int32, device="cuda") for _ in range(2))
            call = lambda: lib.dare_raw(True, 0, N, nX, nU, dA, dB, dQ, dR, dst, K=dK, P=dP, iterations=dit)
            call()
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for e0, e1 in ev:
                e0.record(); call(); e1.record()
            torch.cuda.synchronize()
            ms = float(np.median([e0.elapsed_time(e1) for e0, e1 in ev]))
            st, it = dst.cpu().numpy(), dit.cpu().numpy()
            assert np.all(st == 0), st
            # host path on the same inputs: download, then scipy per model (4096 at 80 x 18: 148 timed, scaled)
            n_host = N if not (nX == 80 and N > 148) else 148
            t0 = time.perf_counter()
            Ah, Bh = dA[:n_host].cpu().numpy(), dB[:n_host].cpu().numpy()
            Kh = host_dare(Ah, Bh, Q, R)
            host_ms = (time.perf_counter() - t0) * 1e3 * N / n_host
            err = float(np.max(np.abs(dK[:n_host].cpu().numpy() - Kh)) / np.max(np.abs(Kh)))
            emit(gpu, row="dare", nX=nX, nU=nU, models=N, device_ms=ms, doublings_max=int(it.max()),
                 doublings_median=float(np.median(it)), host_ms=host_ms, host_models_timed=n_host,
                 speedup=host_ms / ms, max_rel_diff_K_vs_scipy=err)


def end_to_end(gpu, reps):
    import golden_util as G
    d = G.desc("pend_on_cart1")
    refs = [d.param_ref("frame_mass", 3, 0), d.param_ref("frame_value", 3)]
    M = 148
    rng = np.random.default_rng(148)
    vals = np.stack([rng.uniform(0.5, 2.0, M), -rng.uniform(0.5, 1.5, M)], axis=1)
    ds = discopt.DSystem(MV.MidpointVI(d), np.arange(11) * 0.01)
    ds.set_parameters(refs, vals)
    xk, uk = np.array([0.0, np.pi, 0.0, 0.0]), np.zeros(1)
    Q, R = np.diag([10.0, 10.0, 1.0, 1.0]), np.array([[0.1]])
    ds.calc_stationary_controller(xk, uk, Q, R)
    dev_t, host_t = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        K, P = ds.calc_stationary_controller(xk, uk, Q, R)
        dev_t.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        A, B = ds.linearize(np.tile(xk, (M, 1)), np.tile(uk, (M, 1)), np.full(M, 0.0), np.full(M, 0.01),
                            X_hint=np.tile(xk, (M, 1)))
        Kh = host_dare(A, B, Q, R)
        host_t.append(time.perf_counter() - t0)
    err = float(np.max(np.abs(K - Kh)) / np.max(np.abs(Kh)))
    dm, hm = float(np.median(dev_t)) * 1e3, float(np.median(host_t)) * 1e3
    emit(gpu, row="calc_stationary_controller", system="pend_on_cart1", models=M, device_ms=dm,
         host_linearize_then_scipy_ms=hm, speedup=hm / dm, max_rel_diff_K_vs_scipy=err)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    assert lib.device_count() > 0, "time_dare.py needs a CUDA device"
    gpu = card()
    device_rows(gpu, a.reps)
    end_to_end(gpu, a.reps)


if __name__ == "__main__":
    main()
