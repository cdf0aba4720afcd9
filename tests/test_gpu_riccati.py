"""The device Riccati / LQ solve (lqr_kernel behind trepb_lqr_batch* and trepb_lq_batch*) against the long-double
reference of tests/lqref.py, at every shape its launch code branches on (lqr_launch, trepb_lqr.cu):

- 4 x 4 register tiles below nX = 32, with (VEC: nX and nU even) and without 128-bit shared loads; the FP64
  tensor-core products at nX >= 32, and the register tiles there too with TREPB_LQR_NO_MMA=1;
- nU > nX, nX = 1, a single step, ragged tensor-core tiles;
- the largest shapes that fit the shared-memory layout and the in-kernel gamma solve, and the refusals one past them;
- gamma that needs row exchanges, has badly scaled rows or a condition number near 1e8;
- the grid-stride loop over rollouts (batches of twice the resident CTAs and more) with exactly singular rollouts
  between healthy ones in the same CTA;
- the _dev entry point on torch tensors on a non-default stream against the host-array one.

The reference was tied to the original discopt.dlqr through the pinned parity results (test_lq_reference.py)."""
import re

import numpy as np
import pytest

import golden_util as G
import lqref

pytestmark = pytest.mark.gpu

# Well-conditioned random problems (A of spectral radius about 0.9, SPD Q and R): fp64 against long double.
RTOL = 1e-11
EPS = np.finfo(float).eps


@pytest.fixture(scope="module")
def lib():
    from trep_b200 import lib as L
    assert L.device_count() > 0, "GPU tests need a CUDA device"
    return L


@pytest.fixture(scope="module")
def device():
    import torch
    p = torch.cuda.get_device_properties(0)
    return {"optin": p.shared_memory_per_block_optin, "sms": p.multi_processor_count}


# ---- the launch limits, from lqr_launch's sizing ---------------------------------------------------------------

def lqr_smem_bytes(nX, nU):
    """Dynamic shared memory lqr_launch asks for."""
    ldg = (nU + nX + 1) | 1
    return 8 * (3 * nX * nX + 4 * nX * nU + nU * nU + nU * ldg + 4 * nU + 16 + 2 * nX + 2 * nU + 2)


def gj_fits(nX, nU):
    """The elimination deals the nU (nU + nX + 1) elements of [gamma | Kp | c] out to at most 512 threads, 4 each."""
    return nU * (nU + nX + 1) <= 4 * 512


def limit_shapes(optin):
    """The largest supported shapes: nX at nU = 1 (shared memory), nU at nX = 80, 32, 1 (the gamma solve)."""
    nx1 = max(n for n in range(1, 1024) if lqr_smem_bytes(n, 1) <= optin)
    top = lambda nX: max(u for u in range(1, 65) if gj_fits(nX, u))
    out = {"smem_nU1": (nx1, 1), "gj_nX80": (80, top(80)), "gj_nX32": (32, top(32)), "gj_nX1": (1, top(1))}
    for nX, nU in out.values():
        assert lqr_smem_bytes(nX, nU) <= optin and gj_fits(nX, nU)
    return out


def _shape(spec, device):
    return limit_shapes(device["optin"])[spec] if isinstance(spec, str) else spec


def _id(spec):
    return spec if isinstance(spec, str) else "%dx%d" % spec


# ---- problems and comparisons ----------------------------------------------------------------------------------

def _spd(rng, shape, n):
    M = rng.normal(size=shape + (n, n))
    return M @ np.swapaxes(M, -1, -2) / n + np.eye(n)


def problem(rng, N, n, nX, nU):
    """N rollouts of n steps: A of spectral radius about 0.9, B, per-rollout per-step SPD Q [N,n+1] and R [N,n],
    a small cross term S, linear costs q, r."""
    return dict(A=rng.normal(0, 0.9 / np.sqrt(nX), (N, n, nX, nX)), B=rng.normal(size=(N, n, nX, nU)),
                Q=_spd(rng, (N, n + 1), nX), R=_spd(rng, (N, n), nU), S=rng.normal(0, 0.1 / np.sqrt(nX), (N, n, nX, nU)),
                q=rng.normal(size=(N, n + 1, nX)), r=rng.normal(size=(N, n, nU)))


def assert_rollouts_close(got, want, what, rtol=RTOL):
    """golden_util.assert_close on every rollout (axis 0), each against its own max|want|."""
    got, want = np.asarray(got, float), np.asarray(want, float)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    scale = np.max(np.abs(want), axis=tuple(range(1, want.ndim)), keepdims=True)
    bound = rtol * np.abs(want) + G.ATOL_FRAC * (rtol / G.RTOL) * scale
    diff = np.abs(got - want)
    bad = ~(diff <= bound)
    if np.any(bad):
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError("%s: |a-b| = %.3e at %s exceeds %.1e |b| (b = %.3e, max|b| of the rollout = %.3e)"
                             % (what, diff[i], i, rtol, want[i], scale[i[0]].item()))


def ld_batch(p, rows, Q, R, S=None, q=None, r=None, per=False):
    """lqref.solve_tv_lq_ld on rollouts `rows`; the cost arrays shared, or indexed by rollout when per."""
    pick = (lambda x, i: None if x is None else x[i]) if per else (lambda x, i: x)
    outs = [lqref.solve_tv_lq_ld(p["A"][i], p["B"][i], pick(Q, i), pick(R, i), S=pick(S, i), q=pick(q, i),
                                 r=pick(r, i)) for i in rows]
    return [None if o[0] is None else np.stack(o).astype(float) for o in zip(*outs)]


def run_lqr(lib, p, Q, R, with_p0):
    N, n, nX, nU = p["B"].shape
    K, P0, st = np.zeros((N, n, nU, nX)), np.zeros((N, nX, nX)) if with_p0 else None, np.full(N, 7, np.int32)
    lib.lqr_raw(False, 0, N, n, nX, nU, p["A"], p["B"], Q, R, K, st, P0=P0, q_per_step=Q.ndim == 3,
                r_per_step=R.ndim == 3)
    return K, P0, st


def run_lq(lib, A, B, Q, S, R, q, r, per, with_p0):
    N, n, nX, nU = B.shape
    K, Cf, st = np.zeros((N, n, nU, nX)), np.zeros((N, n, nU)), np.full(N, 7, np.int32)
    P0, b0 = (np.zeros((N, nX, nX)), np.zeros((N, nX))) if with_p0 else (None, None)
    lib.lq_raw(False, 0, N, n, nX, nU, A, B, Q, S, R, q, r, K, Cf, st, P0=P0, b0=b0, cost_per_rollout=per)
    return K, Cf, P0, b0, st


LQR_SHAPES = [(1, 1), (2, 2), (4, 2), (6, 4), (3, 5), (2, 9), (31, 2), (32, 2), (33, 3), (47, 7), (64, 8), (81, 3),
              (96, 2), "smem_nU1", "gj_nX80", "gj_nX32", "gj_nX1"]


@pytest.mark.parametrize("nsteps", [1, 2, 13])
@pytest.mark.parametrize("spec", LQR_SHAPES, ids=_id)
def test_riccati_matches_the_long_double_reference(lib, device, monkeypatch, spec, nsteps):
    """Four calls per shape, each against the reference on every rollout:
    LQR with Q, R shared by all steps (with P0), LQR with per-step Q, R (no P0 output), LQ with costs shared by the
    batch and S (with P0, b0), LQ with one cost per rollout and no S (no P0, b0).  At nX >= 32 all four again on the
    register-tile products (TREPB_LQR_NO_MMA=1, read by every launch)."""
    nX, nU = _shape(spec, device)
    N = 2
    p = problem(np.random.default_rng(1000 * nX + 10 * nU + nsteps), N, nsteps, nX, nU)
    Q, R, S, q, r = p["Q"], p["R"], p["S"], p["q"], p["r"]
    rows = range(N)
    want = {
        "lqr shared": ld_batch(p, rows, Q[0, 0], R[0, 0]),
        "lqr per step": ld_batch(p, rows, Q[0], R[0]),
        "lq shared S": ld_batch(p, rows, Q[0], R[0], S[0], q[0], r[0]),
        "lq per rollout": ld_batch(p, rows, Q, R, None, q, r, per=True),
    }
    monkeypatch.delenv("TREPB_LQR_NO_MMA", raising=False)
    for path in ["tensor cores" if nX >= 32 else "register tiles"] + (["register tiles forced"] if nX >= 32 else []):
        if path.endswith("forced"):
            monkeypatch.setenv("TREPB_LQR_NO_MMA", "1")
        got = {
            "lqr shared": run_lqr(lib, p, Q[0, 0], R[0, 0], True),
            "lqr per step": run_lqr(lib, p, Q[0], R[0], False),
            "lq shared S": run_lq(lib, p["A"], p["B"], Q[0], S[0], R[0], q[0], r[0], False, True),
            "lq per rollout": run_lq(lib, p["A"], p["B"], Q, None, R, q, r, True, False),
        }
        for case, out in got.items():
            what = "%dx%d K=%d %s (%s)" % (nX, nU, nsteps, case, path)
            assert np.all(out[-1] == 0), (what, out[-1])
            names = ("K", "P0") if case.startswith("lqr") else ("K", "C", "P0", "b0")
            for name, g, w in zip(names, out[:-1], want[case] if case.startswith("lq ") else
                                  (want[case][0], want[case][2])):
                if g is not None:
                    assert_rollouts_close(g, w, "%s %s" % (what, name))


# ---- conditioning of gamma -------------------------------------------------------------------------------------

def _conditioned(kind, rng, nU):
    """R at the special step (where B = 0, so gamma = R exactly) and the scale of S there."""
    if kind == "row exchanges":
        # indefinite and nonsingular, zero leading diagonal: the first pivot must come from row 1
        R = np.eye(nU); R[:2, :2] = [[0.0, 1.0], [1.0, 0.0]]
        return R, 0.1
    if kind == "badly scaled rows":
        D = np.ones(nU); D[:3] = [1e-6, 1.0, 1e6]
        return D[:, None] * _spd(rng, (), nU), 1e-4
    # a random SPD gamma with condition number 1e8
    U, _ = np.linalg.qr(rng.normal(size=(nU, nU)))
    return (U * np.logspace(0, -8, nU)) @ U.T, 1e-5


@pytest.mark.parametrize("nX,nU", [(6, 4), (5, 3), (40, 4)], ids=["6x4", "5x3", "40x4"])
@pytest.mark.parametrize("kind", ["row exchanges", "badly scaled rows", "kappa 1e8"])
def test_gamma_conditioning_and_pivoting(lib, kind, nX, nU):
    """LQ with shared costs and S over 4 steps; at step 2, B = 0 and R is the conditioned matrix, so gamma = R.

    Tolerance: max(1e-11, 100 eps kappa), kappa the largest condition number of a row-equilibrated gamma (the
    elimination pivots on implicitly row-scaled values, so row scaling alone costs no accuracy).  That is 1e-11 for
    the row exchanges and the scaled rows, about 2e-6 for kappa 1e8."""
    rng = np.random.default_rng(77 + nX)
    N, n, k0 = 2, 4, 2
    p = problem(rng, N, n, nX, nU)
    R, s = _conditioned(kind, rng, nU)
    p["B"][:, k0] = 0.0
    p["R"][0, k0] = R
    p["S"][0, k0] *= s / 0.1 * np.sqrt(nX)
    Q, R, S, q, r = p["Q"][0], p["R"][0], p["S"][0], p["q"][0], p["r"][0]
    gammas = []
    want = [np.stack(w).astype(float) for w in zip(*[lqref.solve_tv_lq_ld(p["A"][i], p["B"][i], Q, R, S=S, q=q, r=r,
                                                                       gammas=gammas) for i in range(N)])]
    kappa = max(np.linalg.cond(g.astype(float) / np.max(np.abs(g.astype(float)), axis=1, keepdims=True))
                for g in gammas)
    rtol = max(RTOL, 100 * EPS * kappa)
    if kind == "kappa 1e8":
        assert kappa > 1e7
    out = run_lq(lib, p["A"], p["B"], Q, S, R, q, r, False, True)
    assert np.all(out[-1] == 0), out[-1]
    for name, g, w in zip(("K", "C", "P0", "b0"), out[:-1], want):
        assert_rollouts_close(g, w, "%s %dx%d %s (kappa %.1e)" % (kind, nX, nU, name, kappa), rtol=rtol)


# ---- limits and refusals ---------------------------------------------------------------------------------------

def _refusal_cases(device):
    lim = limit_shapes(device["optin"])
    nx1 = lim["smem_nU1"][0]
    return {
        "smem_nU1+1": ((nx1 + 1, 1, 1), 4, "state dimension too large for the shared-memory Riccati sweep"),
        "gj_nX80+1": ((80, lim["gj_nX80"][1] + 1, 1), 4, "input dimension too large for the in-kernel gamma solve"),
        "gj_nX1+1": ((1, lim["gj_nX1"][1] + 1, 1), 4, "input dimension too large for the in-kernel gamma solve"),
        # the gamma-solve limit refuses every nU >= 45 before "more than 64 inputs" could; either names the refusal
        "nU65": ((1, 65, 1), 4, "more than 64 inputs|input dimension too large for the in-kernel gamma solve"),
        "nU0": ((3, 0, 2), 1, "bad sizes"),
        "nsteps0": ((3, 2, 0), 1, "bad sizes"),
    }


@pytest.mark.parametrize("case", ["smem_nU1+1", "gj_nX80+1", "gj_nX1+1", "nU65", "nU0", "nsteps0"])
def test_refusals_launch_nothing(lib, device, case):
    """Both _dev entry points refuse with the code and message, and leave every output (filled with a sentinel) as
    it was: nothing ran."""
    import torch
    (nX, nU, n), code, msg = _refusal_cases(device)[case]
    N, m = 2, max(n, 1)
    z = lambda *s: torch.full(s, 0.5, dtype=torch.float64, device="cuda")
    A, B, Q, R, S, q, r = z(N, m, nX, nX), z(N, m, nX, max(nU, 1)), z(m + 1, nX, nX), z(m, max(nU, 1), max(nU, 1)), \
        z(m, nX, max(nU, 1)), z(m + 1, nX), z(m, max(nU, 1))
    outs = dict(K=z(N, m, max(nU, 1), nX), C=z(N, m, max(nU, 1)), P0=z(N, nX, nX), b0=z(N, nX),
                st=torch.full((N,), 7, dtype=torch.int32, device="cuda"))
    before = {k: v.clone() for k, v in outs.items()}
    with pytest.raises(lib.TrepbError) as e:
        lib.lq_raw(True, 0, N, n, nX, nU, A, B, Q, S, R, q, r, outs["K"], outs["C"], outs["st"], P0=outs["P0"],
                   b0=outs["b0"])
    assert e.value.code == code and re.search(msg, str(e.value)), str(e.value)
    with pytest.raises(lib.TrepbError) as e:
        lib.lqr_raw(True, 0, N, n, nX, nU, A, B, Q, R, outs["K"], outs["st"], P0=outs["P0"], q_per_step=True,
                    r_per_step=True)
    assert e.value.code == code and re.search(msg, str(e.value)), str(e.value)
    torch.cuda.synchronize()
    for k, v in outs.items():
        assert torch.equal(v, before[k]), k


# ---- the grid-stride loop over rollouts, with singular ones ----------------------------------------------------

@pytest.mark.parametrize("nX,nU,n", [(4, 2, 6), (80, 18, 3)], ids=["4x2", "80x18"])
def test_grid_stride_batch_with_singular_rollouts(lib, device, nX, nU, n):
    """One cost per rollout and S; every 97th rollout (0 among them) is exactly singular at step 1 (R = 0, B = 0).
    The batch exceeds twice the resident CTAs (80x18: one 512-thread CTA per SM; 4x2: a generous 10000), so CTAs
    solve several rollouts each and failing rollouts precede healthy ones in the same CTA."""
    N = 2 * device["sms"] + 3 if nX >= 32 else 10000
    rng = np.random.default_rng(5 + nX)
    p = problem(rng, N, n, nX, nU)
    bad = np.arange(N) % 97 == 0
    p["R"][bad, 1] = 0.0
    p["B"][bad, 1] = 0.0
    A, B, Q, S, R, q, r = (p[k] for k in "ABQSRqr")
    K, Cf, P0, b0, st = run_lq(lib, A, B, Q, S, R, q, r, True, True)
    assert np.array_equal(st, np.where(bad, -2, 0)), np.flatnonzero(st != np.where(bad, -2, 0))[:10]
    ok = ~bad
    want = lqref.solve_tv_lq_f64(A[ok], B[ok], Q[ok], R[ok], S=S[ok], q=q[ok], r=r[ok])
    for name, g, w in zip(("K", "C", "P0", "b0"), (K, Cf, P0, b0), want):
        assert_rollouts_close(g[ok], w, "%dx%d batch %d %s vs fp64" % (nX, nU, N, name))
    # a sample of healthy rollouts, spread over the batch and both ends: long double, and the same bits alone
    healthy = np.flatnonzero(ok)
    sample = np.unique(np.concatenate([healthy[G.rows(len(healthy), 16)], [1, N - 1]]))
    assert len(sample) >= 16
    want = ld_batch(p, sample, Q, R, S, q, r, per=True)
    for name, g, w in zip(("K", "C", "P0", "b0"), (K, Cf, P0, b0), want):
        assert_rollouts_close(g[sample], w, "%dx%d batch %d %s vs long double" % (nX, nU, N, name))
    for i in sample:
        s = slice(i, i + 1)
        one = run_lq(lib, *(np.ascontiguousarray(x[s]) for x in (A, B, Q, S, R, q, r)), True, True)
        for name, g, w in zip(("K", "C", "P0", "b0", "status"), one, (K, Cf, P0, b0, st)):
            assert g.tobytes() == w[s].tobytes(), "rollout %d alone: %s" % (i, name)
    with pytest.raises(lib.TrepbError) as e:
        lib.solve_tv_lq(A, B, q, r, Q, S, R)
    named = [int(x) for x in re.search(r"rollout\(s\) \[([^\]]*)\]", str(e.value)).group(1).split()]
    assert named == list(np.flatnonzero(bad)[:8]), str(e.value)


# ---- the entry points ------------------------------------------------------------------------------------------

@pytest.mark.parametrize("nX,nU", [(6, 4), (64, 8)], ids=["6x4-register-tiles", "64x8-tensor-cores"])
def test_dev_entry_points_on_torch_tensors_give_the_host_bits(lib, monkeypatch, nX, nU):
    """trepb_lq_batch_dev / trepb_lqr_batch_dev on torch tensors, launched on a non-default stream, against
    trepb_lq_batch / trepb_lqr_batch with host arrays: the same bits."""
    import torch
    monkeypatch.delenv("TREPB_LQR_NO_MMA", raising=False)
    N, n = 5, 7
    p = problem(np.random.default_rng(11), N, n, nX, nU)
    A, B, Q, S, R, q, r = (p[k] for k in "ABQSRqr")
    host = run_lq(lib, A, B, Q, S, R, q, r, True, True)
    host_lqr = run_lqr(lib, p, Q[0], R[0], True)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    stream = torch.cuda.Stream()
    dK, dC, dP, db = (torch.full(x.shape, np.nan, dtype=torch.float64, device="cuda") for x in host[:4])
    dst = torch.full((N,), 7, dtype=torch.int32, device="cuda")
    lK, lP = torch.full(host_lqr[0].shape, np.nan, dtype=torch.float64, device="cuda"), \
        torch.full(host_lqr[1].shape, np.nan, dtype=torch.float64, device="cuda")
    lst = torch.full((N,), 7, dtype=torch.int32, device="cuda")
    ins = [t(x) for x in (A, B, Q, S, R, q, r, Q[0], R[0])]
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        lib.lq_raw(True, 0, N, n, nX, nU, *ins[:7], dK, dC, dst, P0=dP, b0=db, cost_per_rollout=True,
                   stream=stream.cuda_stream)
        lib.lqr_raw(True, 0, N, n, nX, nU, ins[0], ins[1], ins[7], ins[8], lK, lst, P0=lP, q_per_step=True,
                    r_per_step=True, stream=stream.cuda_stream)
    stream.synchronize()
    for name, d, h in zip(("K", "C", "P0", "b0", "status"), (dK, dC, dP, db, dst), host):
        assert d.cpu().numpy().tobytes() == h.tobytes(), "lq " + name
    for name, d, h in zip(("K", "P0", "status"), (lK, lP, lst), host_lqr):
        assert d.cpu().numpy().tobytes() == h.tobytes(), "lqr " + name
