"""Closed-loop cost and stability of stationary gains: the Lyapunov solve on the device (trepb_dlyap_batch_dev) against
the host path it replaces.

  device:      CUDA events around the _dev call (inputs already in HBM), median of `reps` after one warm-up, at the
               pend-on-cart's dims (4 x 1) and the marionette's (80 x 18), for 1, 148 and 4096 pairs.  The pairs are
               random stable closed loops (tests/test_gpu_dlyap.py's generator, spectral radius 0.9); the doubling
               steps taken are reported with the time.
  host:        what a user does without it: download A / B / K from the device, then form A_c, Q_c and call
               scipy.linalg.solve_discrete_lyapunov once per pair (host clock, one pass; 4096 pairs at 80 x 18 are
               timed on 148 and scaled).
  end to end:  DSystem.evaluate_stationary_controller on pend-on-cart at the upright equilibrium, 64 gains (one DARE
               gain per model) under 64 models (set_parameters): upload, linearize, 4096 Lyapunov solves,
               synchronize, download cost and status (host clock, median of reps), against DSystem.linearize followed
               by the host path over the same 64 x 64 pairs.

Usage: python tools/time_dlyap.py [--reps 20]
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
PAIRS = [1, 148, 4096]


def emit(gpu, **row):
    print(json.dumps(dict(row, card=gpu[0], power_limit=gpu[1])), flush=True)


def host_dlyap(A, B, K, Q, R, gi, mi):
    """cost trace(P) per pair, scipy on the host."""
    import scipy.linalg as sla
    out = np.empty(len(gi))
    for p, (g, m) in enumerate(zip(gi, mi)):
        Ac = A[m] - B[m] @ K[g]
        P = sla.solve_discrete_lyapunov(Ac.T, Q + K[g].T @ R @ K[g])
        out[p] = np.trace(P)
    return out


def device_rows(gpu, reps):
    import torch
    from test_gpu_dlyap import closed_loop_problem
    for nX, nU in SHAPES:
        for N in PAIRS:
            A, B, K, Q, R, _ = closed_loop_problem(np.random.default_rng(N + nX), N, nX, nU)
            t = lambda x: torch.tensor(np.ascontiguousarray(x), device="cuda")
            dA, dB, dK, dQ, dR, dW = t(A), t(B), t(K), t(Q), t(R), t(np.eye(nX))
            dc = torch.empty(N, dtype=torch.float64, device="cuda")
            dst, dit = (torch.empty(N, dtype=torch.int32, device="cuda") for _ in range(2))
            call = lambda: lib.dlyap_raw(True, 0, N, N, N, nX, nU, dA, dB, dK, dQ, dR, dst, W=dW, cost=dc,
                                         iterations=dit)
            call()
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for e0, e1 in ev:
                e0.record(); call(); e1.record()
            torch.cuda.synchronize()
            ms = float(np.median([e0.elapsed_time(e1) for e0, e1 in ev]))
            st, it = dst.cpu().numpy(), dit.cpu().numpy()
            assert np.all(st == 0), st
            # host path on the same inputs: download, then scipy per pair (4096 at 80 x 18: 148 timed, scaled)
            n_host = N if not (nX == 80 and N > 148) else 148
            t0 = time.perf_counter()
            Ah, Bh, Kh = dA[:n_host].cpu().numpy(), dB[:n_host].cpu().numpy(), dK[:n_host].cpu().numpy()
            ch = host_dlyap(Ah, Bh, Kh, Q, R, np.arange(n_host), np.arange(n_host))
            host_ms = (time.perf_counter() - t0) * 1e3 * N / n_host
            err = float(np.max(np.abs(dc[:n_host].cpu().numpy() - ch) / np.abs(ch)))
            emit(gpu, row="dlyap", nX=nX, nU=nU, pairs=N, device_ms=ms, doublings_max=int(it.max()),
                 doublings_median=float(np.median(it)), host_ms=host_ms, host_pairs_timed=n_host,
                 speedup=host_ms / ms, max_rel_diff_cost_vs_scipy=err)


def end_to_end(gpu, reps):
    import golden_util as G
    d = G.desc("pend_on_cart1")
    refs = [d.param_ref("frame_mass", 3, 0), d.param_ref("frame_value", 3)]
    M = 64
    rng = np.random.default_rng(4096)
    vals = np.stack([rng.uniform(0.5, 2.0, M), -rng.uniform(0.5, 1.5, M)], axis=1)
    ds = discopt.DSystem(MV.MidpointVI(d), np.arange(11) * 0.01)
    ds.set_parameters(refs, vals)
    xk, uk = np.array([0.0, np.pi, 0.0, 0.0]), np.zeros(1)
    Q, R = np.diag([100.0, 100.0, 1.0, 1.0]), np.array([[0.01]])
    K, _ = ds.calc_stationary_controller(xk, uk, Q, R)
    ds.evaluate_stationary_controller(xk, uk, K, Q, R)
    gi, mi = np.repeat(np.arange(M), M), np.tile(np.arange(M), M)
    dev_t, host_t = [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        cost, st = ds.evaluate_stationary_controller(xk, uk, K, Q, R)
        dev_t.append(time.perf_counter() - t0)
    for _ in range(max(1, reps // 5)):
        t0 = time.perf_counter()
        A, B = ds.linearize(np.tile(xk, (M, 1)), np.tile(uk, (M, 1)), np.full(M, 0.0), np.full(M, 0.01),
                            X_hint=np.tile(xk, (M, 1)))
        ch = host_dlyap(A, B, K, Q, R, gi, mi)
        host_t.append(time.perf_counter() - t0)
    ch = ch.reshape(M, M)
    stable = st == 0
    err = float(np.max(np.abs(cost[stable] - ch[stable]) / np.abs(ch[stable])))
    dm, hm = float(np.median(dev_t)) * 1e3, float(np.median(host_t)) * 1e3
    emit(gpu, row="evaluate_stationary_controller", system="pend_on_cart1", gains=M, models=M, device_ms=dm,
         host_linearize_then_scipy_ms=hm, host_reps=len(host_t), speedup=hm / dm, stable_pairs=int(stable.sum()),
         max_rel_diff_cost_vs_scipy=err)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    assert lib.device_count() > 0, "time_dlyap.py needs a CUDA device"
    gpu = card()
    device_rows(gpu, a.reps)
    end_to_end(gpu, a.reps)


if __name__ == "__main__":
    main()
