"""Batched mirror of the reference's ``trep.MidpointVI`` Python shell (trep/midpointvi.py:19-732).

Same method names, argument meaning and error behaviour; every state array gains a leading batch
axis (``q1`` is ``[B, nq]`` ...).  All numerics run in the CUDA library through the C ABI
(``trep_b200.lib``) - there is no CPU path.

    mvi = MidpointVI(system)                      # model mirror, SystemDesc or a live trep.System
    mvi.initialize_from_configs(0.0, q0, dt, q1)  # [B, nq] each
    iters = mvi.step(mvi.t2 + dt, u1, k2)         # one DEL step for every instance
    mvi.simulate(1000, dt)                        # many steps inside one kernel launch
"""
from __future__ import annotations

import numpy as np

from . import desc as D
from . import lib, model


class ConvergenceError(Exception):
    """Mirror of trep.ConvergenceError (trep/_trep/_trep.c:142): raised when at least one instance
    failed; ``.status`` holds the per-instance codes (0 ok, -1 not converged, -2 singular)."""

    def __init__(self, msg, status):
        super().__init__(msg)
        self.status = status


def as_desc(system) -> D.SystemDesc:
    if isinstance(system, D.SystemDesc):
        return system
    if isinstance(system, model.System):
        return system.describe()
    return model.flatten_trep_system(system)   # live reference trep.System (duck-typed)


class MidpointVI:
    def __init__(self, system, tolerance=1e-10, device=0, specialize=True):
        self.desc = as_desc(system)
        # coop_varied: set_parameters works on a cooperative handle too (the marionette's); plain calls are unchanged
        self.sys = lib.System(self.desc, device=device, specialize=specialize, coop_varied=True)
        self.tolerance = float(tolerance)
        d = self.desc
        self.nq, self.nd, self.nk, self.nu, self.nc = d.nq, d.nd, d.nk, d.nu, d.nc
        self.t1 = self.t2 = 0.0
        self.q1 = self.q2 = self.p1 = self.p2 = self.u1 = self.lambda1 = None
        self.status = None
        self._lin = None
        self._d2 = None
        self._params = None

    def set_parameters(self, refs, values):
        """Per-instance physical parameters for every later initialize_from_*, step, simulate, calc_f,
        discrete_fm2 and first-derivative call: refs a list of SystemDesc.param_ref entries, values [B][len(refs)]
        (instance b runs on row b).  set_parameters(None, None) goes back to the description's numbers.  The
        second-derivative getters raise while parameters are set (lib.System.deriv2(params=...) and
        DSystem.set_parameters take per-instance parameters)."""
        if refs is None:
            self._params = None
        else:
            refs = [tuple(r) for r in refs]
            lib.check_params(self.desc, refs)
            values = np.ascontiguousarray(np.asarray(values, dtype=np.float64).reshape(-1, len(refs)))
            self._params = (refs, values)
        self._lin = None
        self._d2 = None

    def _p(self, B):
        if self._params is not None and self._params[1].shape[0] != B:
            raise ValueError("parameters have %d rows for a batch of %d" % (self._params[1].shape[0], B))
        return self._params

    # ---- initialisation (midpointvi.py:138-172) --------------------------------------------------
    def _b(self, x, n):
        x = np.asarray(x, dtype=np.float64)
        if x.ndim == 1:
            x = x[None, :]
        assert x.shape[1] == n, "expected trailing dimension %d, got %r" % (n, x.shape)
        return np.ascontiguousarray(x)

    def initialize_from_state(self, t1, q1, p1, lambda1=None):
        self.q1 = self.q2 = self._b(q1, self.nq)
        self.p1 = self.p2 = self._b(p1, self.nd)
        self.t1 = self.t2 = float(t1)
        B = self.q1.shape[0]
        self.lambda1 = np.zeros((B, self.nc)) if lambda1 is None else self._b(lambda1, self.nc)
        self._lin = None
        self._d2 = None

    def initialize_from_configs(self, t0, q0, t1, q1, lambda1=None):
        q0, q1 = self._b(q0, self.nq), self._b(q1, self.nq)
        self.t1, self.t2 = float(t0), float(t1)
        self.q1, self.q2 = q0, q1
        self.p2 = self.sys.calc_p2(self.t2 - self.t1, q0, q1, params=self._p(q1.shape[0]))
        self.p1 = None
        B = q1.shape[0]
        self.lambda1 = np.zeros((B, self.nc)) if lambda1 is None else self._b(lambda1, self.nc)
        self._lin = None
        self._d2 = None

    @property
    def batch(self):
        return 0 if self.q2 is None else self.q2.shape[0]

    # ---- stepping (midpointvi.py:174-201) ---------------------------------------------------------
    def _check(self, status):
        self.status = status
        bad = np.flatnonzero(status != 0)
        if bad.size:
            raise ConvergenceError("%d of %d instances failed (first: instance %d, status %d) at t=%s"
                                   % (bad.size, status.size, bad[0], status[bad[0]], self.t2), status)

    def step(self, t2, u1=tuple(), k2=tuple(), max_iterations=200, q2_hint=None, lambda1_hint=None):
        """Advance every instance to time t2.  Returns the per-instance Newton iteration counts."""
        B = self.batch
        u1 = np.broadcast_to(np.asarray(u1, float).reshape(-1, self.nu) if self.nu else np.zeros((1, 0)), (B, self.nu))
        k2 = np.broadcast_to(np.asarray(k2, float).reshape(-1, self.nk) if self.nk else np.zeros((1, 0)), (B, self.nk))
        self.q1, self.p1, self.u1 = self.q2, self.p2, np.ascontiguousarray(u1)
        self.t1, t0 = self.t2, self.t2
        hint = None if q2_hint is None else self._b(q2_hint, np.asarray(q2_hint).shape[-1])[:, :self.nd]
        lam = self.lambda1 if lambda1_hint is None else self._b(lambda1_hint, self.nc)
        out = self.sys.step(self.q1, self.p1, t0, float(t2) - t0, nsteps=1,
                            u1=u1[:, None, :] if self.nu else None, k2=k2[:, None, :] if self.nk else None,
                            q2_guess=hint, lambda_guess=lam if self.nc else None,
                            tolerance=self.tolerance, max_iterations=max_iterations, params=self._p(B))
        self.t2 = float(t2)
        self.q2, self.p2, self.lambda1 = out["q2"], out["p2"], out["lambda1"]
        self._lin = None
        self._d2 = None
        self._check(out["status"])
        return out["iters"]

    def simulate(self, nsteps, dt, u=None, k=None, max_iterations=200, sample_every=0, times=None, params=None):
        """`nsteps` steps inside one kernel launch (the Monte-Carlo / rollout path): of length dt, or on
        the grid `times` [nsteps+1] (times[0] = the current t2; any spacing).
        u: [B, nsteps, nu], k: [B, nsteps, nk] (kinematic configs at the END of each step).
        params: (refs, values [B][len(refs)]) for this call only, instead of set_parameters' (ValueError when both
        are set); the state it leaves was reached on those rows, later calls run on set_parameters' again.
        Returns dict(iters, traj_q, traj_p) - trajectories only if sample_every > 0."""
        if params is not None and self._params is not None:
            raise ValueError("parameters are set on this MidpointVI and passed to simulate: clear one of them")
        if params is not None:
            refs = [tuple(r) for r in params[0]]
            params = (refs, np.ascontiguousarray(np.asarray(params[1], dtype=np.float64).reshape(self.batch, len(refs))))
        out = self.sys.step(self.q2, self.p2, self.t2, float(dt), nsteps=nsteps, u1=u, k2=k,
                            lambda_guess=self.lambda1 if self.nc else None, tolerance=self.tolerance,
                            max_iterations=max_iterations, sample_every=sample_every, times=times,
                            params=self._p(self.batch) if params is None else params)
        # state before the last step is only known when a trajectory was captured
        self.q1 = self.p1 = None
        t = self.t2
        if times is not None:
            self.t1, t = float(times[-2]), float(times[-1])
        else:
            for _ in range(nsteps):       # same accumulation as repeated step(t2 + dt) calls
                self.t1, t = t, t + float(dt)
        self.t2 = t
        self.q2, self.p2, self.lambda1 = out["q2"], out["p2"], out["lambda1"]
        self._lin = None
        self._d2 = None
        self._check(out["status"])
        return out

    def calc_f(self):
        """Residual of the DEL equation at the current (q1, q2, p1, u1, lambda1): [B, nd+nc]
        (_MidpointVI._calc_f, midpointvi.c:567-575)."""
        assert self.q1 is not None and self.p1 is not None, "calc_f needs the state before the step"
        return self.sys.calc_f(self.t1, self.t2, self.q1, self.q2, self.p1, self.u1, self.lambda1 if self.nc else None,
                               params=self._p(self.batch))

    def discrete_fm2(self):
        """Discrete forcing of the current step [B, nd] (_MidpointVI.discrete_fm2, midpointvi.c:2710-2727)."""
        assert self.q1 is not None, "discrete_fm2 needs the configuration before the step"
        return self.sys.discrete_fm2(self.t1, self.t2, self.q1, self.q2, self.u1, params=self._p(self.batch))

    @property
    def v2(self):
        """Discrete kinematic velocity (q2k - q1k)/(t2 - t1)  (midpointvi.py:325-333)."""
        if self.t2 != self.t1 and self.q1 is not None:
            return ((self.q2 - self.q1) / (self.t2 - self.t1))[:, self.nd:]
        return None

    # ---- first derivatives (midpointvi.py:337-420): getters return [B, out, wrt] ---------------------
    def _calc_deriv1(self):
        if self._lin is None:
            assert self.q1 is not None and self.p1 is not None, "derivatives need the state before the step"
            out = self.sys.linearize(self.q1, self.p1, self.u1, self.q2[:, self.nd:], t1=self.t1, t2=self.t2,
                                     q2_guess=self.q2[:, :self.nd], lambda_guess=self.lambda1 if self.nc else None,
                                     want_raw=True, tolerance=self.tolerance, params=self._p(self.batch))
            self._check(out["status"])
            self._lin = out
        return self._lin

    def _get(self, name):
        return np.ascontiguousarray(np.swapaxes(self._calc_deriv1()[name], 1, 2))

    def q2_dq1(self): return self._get("q2_dq1")
    def q2_dp1(self): return self._get("q2_dp1")
    def q2_du1(self): return self._get("q2_du1")
    def q2_dk2(self): return self._get("q2_dk2")
    def p2_dq1(self): return self._get("p2_dq1")
    def p2_dp1(self): return self._get("p2_dp1")
    def p2_du1(self): return self._get("p2_du1")
    def p2_dk2(self): return self._get("p2_dk2")
    def lambda1_dq1(self): return self._get("l1_dq1")
    def lambda1_dp1(self): return self._get("l1_dp1")
    def lambda1_du1(self): return self._get("l1_du1")
    def lambda1_dk2(self): return self._get("l1_dk2")

    # ---- second derivatives (midpointvi.py:422-731): the 30 tensors in the reference's storage layout
    #      [B][wrt A][wrt B][out]  (trep.h:439-473), e.g. q2_dq1dq1()[b, i, j, :] = d2 q2 / dq1_i dq1_j
    def _calc_deriv2(self):
        if self._params is not None:
            raise NotImplementedError("MidpointVI's second-derivative getters have no per-instance-parameter form: "
                                      "call set_parameters(None, None) first, or use lib.System.deriv2(params=...) "
                                      "or DSystem.set_parameters")
        if getattr(self, "_d2", None) is None or self._lin is None:
            assert self.q1 is not None and self.p1 is not None, "derivatives need the state before the step"
            out = self.sys.deriv2(self.q1, self.p1, self.u1, self.q2[:, self.nd:], t1=self.t1, t2=self.t2,
                                  q2_guess=self.q2[:, :self.nd], lambda_guess=self.lambda1 if self.nc else None,
                                  tolerance=self.tolerance)
            self._check(out["status"])
            self._lin = out
            self._d2 = out
        return self._d2

    def __getattr__(self, name):
        # q2_dq1dq1 ... p2_dk2dk2, lambda1_dq1dq1 ... : getters generated from the tensor names
        base = name.replace("lambda1_", "l1_", 1)
        which, _, kind = base.partition("_")
        if which in ("q2", "p2", "l1") and len(kind) == 6 and kind[:3] in ("dq1", "dp1", "du1", "dk2") \
                and kind[3:] in ("dq1", "dp1", "du1", "dk2"):
            def getter():
                d2 = self._calc_deriv2()
                if base in d2:
                    return d2[base]
                # the mirrored block (e.g. dp1dq1) is the transpose of the stored one (dq1dp1)
                return np.ascontiguousarray(np.swapaxes(d2[which + "_" + kind[3:] + kind[:3]], 1, 2))
            return getter
        raise AttributeError(name)


def monte_carlo_sweep(system, q0, dt, nsteps, q1=None, u=None, k=None, tolerance=1e-10, device=None, group=None,
                      hist_max=8, params=None):
    """Monte-Carlo initial-condition sweep (BASELINE.json config 4): every row of q0 [N, nq] is an
    independent rollout started with ``initialize_from_configs(0, q0, dt, q1 or q0)`` and stepped
    ``nsteps`` times inside one kernel launch.  With a ``trep_b200.dist.Group`` (one process per GPU) the
    rollouts are block-partitioned over the ranks - no exchange while stepping - and only the final
    states (q2, p2: 8 (nq + nd) bytes per rollout), the per-rollout iteration totals and status codes
    are gathered on rank 0, device to device (NCCL).  Returns dict(q2 [N,nq], p2 [N,nd], iters [N],
    status [N], hist) on rank 0 (None elsewhere): ``hist[i]`` = number of rollouts whose mean Newton
    iterations per step rounds to i.  params=(refs, values [N][len(refs)]): per-rollout physical parameters
    (SystemDesc.param_ref entries), sharded like q0."""
    from . import dist as D_
    q0 = np.atleast_2d(np.asarray(q0, float))
    n = q0.shape[0]
    world = 1 if group is None else group.world
    rank = 0 if group is None else group.rank
    if device is None:
        device = 0 if group is None else group.device
    lo, hi = D_.shard_range(n, rank, world)
    sl = slice(lo, hi)
    q1s = q0[sl] if q1 is None else np.atleast_2d(np.asarray(q1, float))[sl]
    us = None if u is None else np.asarray(u, float)[sl]
    ks = None if k is None else np.asarray(k, float)[sl]
    mvi = MidpointVI(system, tolerance=tolerance, device=device)
    cnt = hi - lo
    ps = None
    if params is not None:
        refs = [tuple(r) for r in params[0]]
        ps = (refs, np.ascontiguousarray(np.asarray(params[1], float).reshape(n, len(refs))[sl]))
        mvi.set_parameters(*ps)
    if world == 1:
        mvi.initialize_from_configs(0.0, q0[sl], dt, q1s)
        out = mvi.sys.step(mvi.q2, mvi.p2, mvi.t2, float(dt), nsteps=nsteps, u1=us, k2=ks, tolerance=tolerance, params=ps)
        q2, p2, iters, status = out["q2"], out["p2"], out["iters"], out["status"]
    else:
        s, nq, nd = mvi.sys, mvi.nq, mvi.nd
        up = lambda a: lib.DeviceBuffer(device, a.shape, np.float64).upload(np.ascontiguousarray(a, dtype=np.float64))
        dq0, dq1 = up(q0[sl]), up(q1s)
        du = None if us is None or not mvi.nu else up(us)
        dk = None if ks is None or not mvi.nk else up(ks)
        m = max(cnt, 1)
        dp = lib.DeviceBuffer(device, (m, nd)); q2d = lib.DeviceBuffer(device, (m, nq)); p2d = lib.DeviceBuffer(device, (m, nd))
        itd = lib.DeviceBuffer(device, (m,), np.int32); std = lib.DeviceBuffer(device, (m,), np.int32)
        dv = None if ps is None else (ps[0], up(ps[1]) if cnt else None)
        s.calc_p2_raw(True, cnt, float(dt), dq0, dq1, dp, params=dv)
        s.step_raw(True, cnt, nsteps, float(dt), float(dt), dq1, dp, du, dk, None, None, q2d, p2d, None, itd, std,
                   tolerance=tolerance, params=dv)
        res = []
        for buf, rb, dt_, shape in ((q2d, 8 * nq, np.float64, (n, nq)), (p2d, 8 * nd, np.float64, (n, nd)),
                                    (itd, 4, np.int32, (n,)), (std, 4, np.int32, (n,))):
            full = D_.gather_rows(buf, cnt, n, rb, group.comm, device)
            res.append(None if full is None else full.download()[:n * rb].view(dt_).reshape(shape).copy())
            if full is not None:
                full.free()
        for b in (dq0, dq1, du, dk, dp, q2d, p2d, itd, std, None if dv is None else dv[1]):
            if b is not None:
                b.free()
        if rank != 0:
            return None
        q2, p2, iters, status = res
    mean = np.rint(iters[status == 0] / float(nsteps)).astype(np.int64)
    hist = np.bincount(np.clip(mean, 0, hist_max), minlength=hist_max + 1)
    return dict(q2=q2, p2=p2, iters=iters, status=status, hist=hist)
