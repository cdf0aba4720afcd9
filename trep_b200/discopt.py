"""Batched mirror of the part of ``trep.discopt.DSystem`` that sits on the hot path
(trep/discopt/dsystem.py:19-66 state layout, :229-250 set, :284-317 fdx/fdu, :406-423
linearize_trajectory).

State / input layout is the reference's:  X = [Q(nq); p(nd); v(nk)],  U = [u(nu); rho(nk)].

``linearize_trajectory`` treats every time-step k (and every rollout) as an independent instance -
exactly what the reference's loop does (it *sets* the state at every k, dsystem.py:413-415) - and
evaluates all of them in one kernel launch.  With a ``trep_b200.dist.Group`` (one process per GPU) the
instances are block-partitioned over the ranks and the A / B slabs are collected on rank 0 device to
device over NVLink - by NCCL, or by the linearize kernel itself writing into rank 0's peer-mapped slab
(the only exchange this path has; SURVEY.md 8e).
"""
from __future__ import annotations

from collections import namedtuple

import numpy as np

from .midpointvi import ConvergenceError, MidpointVI


from .dist import shard_range  # noqa: F401  (re-exported: the block partition of the instances)


class DSystem:
    linearization_return = namedtuple("linearization", "A B")
    trajectory_return = namedtuple("trajectory", "X U")

    def __init__(self, varint: MidpointVI, t):
        self.varint = varint
        self._time = np.array(t, dtype=np.float64).squeeze()
        v = varint
        self._nQ, self._np, self._nv, self._nu, self._nrho = v.nq, v.nd, v.nk, v.nu, v.nk
        self._nX = self._nQ + self._np + self._nv
        self._nU = self._nu + self._nrho
        self._params = None

    nX = property(lambda s: s._nX)
    nU = property(lambda s: s._nU)
    time = property(lambda s: s._time)

    def kf(self):
        return len(self._time) - 1

    # ---- per-rollout physical parameters -----------------------------------------------------------------
    def set_parameters(self, refs, values):
        """Physical parameters per rollout for robust trajectory optimisation over several plausible models: refs a
        list of SystemDesc.param_ref entries, values [R][len(refs)] (one row per rollout) or one row ([n] / [1, n])
        for every rollout and instance.  set_parameters(None, None) goes back to the description's numbers.
        Trajectory-level calls with R rollouts (linearize_trajectory, calc_feedback_controller, calc_newton_model,
        project, simulate) run rollout r on row r at every step; instance-level calls (f, linearize,
        second_derivatives) take one row per instance; the check_* helpers need a single row.  Any other row count
        raises ValueError."""
        if refs is None:
            self._params = None
            return
        from . import lib
        refs = [tuple(r) for r in refs]
        lib.check_params(self.varint.desc, refs)
        values = np.asarray(values, dtype=np.float64)
        if values.ndim > 2 or values.size == 0 or values.shape[-1] != len(refs):
            raise ValueError("parameter values must be [R][%d] or [%d]" % (len(refs), len(refs)))
        self._params = (refs, np.ascontiguousarray(values.reshape(-1, len(refs))))

    def _rows(self, n, per=1):
        """(refs, values [n][len(refs)]) for n instances, consecutive runs of `per` instances sharing a row (the steps
        of one rollout), or None without parameters."""
        if self._params is None:
            return None
        refs, V = self._params
        if V.shape[0] == 1:
            return refs, np.ascontiguousarray(np.repeat(V, n, axis=0))
        if V.shape[0] * per != n:
            raise ValueError("parameters have %d rows; this call needs %s or a single row"
                             % (V.shape[0], "%d (one per instance)" % n if per == 1 else
                                "%d (one per rollout)" % (n // per)))
        return refs, (V if per == 1 else np.ascontiguousarray(np.repeat(V, per, axis=0)))

    # ---- state packing (dsystem.py:118-226) -----------------------------------------------------------
    def build_state(self, Q=None, p=None, v=None):
        parts = [x for x in (Q, p, v) if x is not None]
        lead = np.asarray(parts[0]).shape[:-1] if parts else ()
        X = np.zeros(lead + (self._nX,))
        if Q is not None: X[..., :self._nQ] = Q
        if p is not None: X[..., self._nQ:self._nQ + self._np] = p
        if v is not None: X[..., self._nQ + self._np:] = v
        return X

    def build_input(self, u=None, rho=None):
        parts = [x for x in (u, rho) if x is not None]
        lead = np.asarray(parts[0]).shape[:-1] if parts else ()
        U = np.zeros(lead + (self._nU,))
        if u is not None: U[..., :self._nu] = u
        if rho is not None: U[..., self._nu:] = rho
        return U

    def split_state(self, X):
        X = np.asarray(X)
        return X[..., :self._nQ], X[..., self._nQ:self._nQ + self._np], X[..., self._nQ + self._np:]

    def split_input(self, U):
        U = np.asarray(U)
        return U[..., :self._nu], U[..., self._nu:]

    def build_trajectory(self, Q=None, p=None, v=None, u=None, rho=None):
        """(X, U) from component trajectories (dsystem.py:140-183); one trajectory ([K+1,.] / [K,.]) or
        a batch with a leading axis.  Unspecified components are zero; lengths are checked against the
        time base like the reference does."""
        K1 = len(self._time)
        lead = ()
        for name, val, n in (("Q", Q, K1), ("p", p, K1), ("v", v, K1), ("u", u, K1 - 1), ("rho", rho, K1 - 1)):
            if val is not None:
                a = np.asarray(val)
                if a.shape[-2] != n:
                    raise ValueError("Invalid length for %s (expected %d)" % (name, n))
                lead = a.shape[:-2]
        X = np.zeros(lead + (K1, self._nX))
        U = np.zeros(lead + (K1 - 1, self._nU))
        if Q is not None: X[..., :self._nQ] = Q
        if p is not None: X[..., self._nQ:self._nQ + self._np] = p
        if v is not None: X[..., self._nQ + self._np:] = v
        if u is not None: U[..., :self._nu] = u
        if rho is not None: U[..., self._nu:] = rho
        return self.trajectory_return(X, U)

    def split_trajectory(self, X=None, U=None):
        """(Q, p, v, u, rho) of a state / input trajectory (dsystem.py:207-226)."""
        Q = p = v = u = rho = None
        if X is not None:
            Q, p, v = self.split_state(X)
        if U is not None:
            u, rho = self.split_input(U)
        return Q, p, v, u, rho

    def save_state_trajectory(self, filename, X=None, U=None):
        """dsystem.py:388-393: the reference's MATLAB trajectory file (batches get a leading axis)."""
        from . import trajectory
        Q, p, v, u, rho = self.split_trajectory(X, U)
        trajectory.save_trajectory(filename, self.varint.desc, self._time, Q, p, v, u, rho)

    def load_state_trajectory(self, filename):
        """dsystem.py:396-402: sets the time base from the file and returns (X, U)."""
        from . import trajectory
        t, Q, p, v, u, rho = trajectory.load_trajectory(filename, self.varint.desc)
        self._time = np.array(t, dtype=np.float64).squeeze()
        return self.build_trajectory(Q, p, v, u, rho)

    def convert_trajectory(self, dsys_a, X, U):
        """Map a trajectory of ``dsys_a`` onto this system by matching config / input names
        (dsystem.py:497-534); components without a counterpart stay zero."""
        a, b = dsys_a.varint.desc, self.varint.desc
        X, U = np.asarray(X, float), np.asarray(U, float)
        qa, pa, va, ua, ra = dsys_a.split_trajectory(X, U)
        nX = np.zeros(X.shape[:-1] + (self._nX,))
        nU = np.zeros(U.shape[:-1] + (self._nU,))
        qb, pb, vb = nX[..., :self._nQ], nX[..., self._nQ:self._nQ + self._np], nX[..., self._nQ + self._np:]
        ub, rb = nU[..., :self._nu], nU[..., self._nu:]

        def copy(dst, src, names_b, names_a):
            for i, n in enumerate(names_b):
                if n in names_a:
                    dst[..., i] = src[..., names_a.index(n)]

        ca, cb = list(a.config_names), list(b.config_names)
        copy(qb, qa, cb, ca)
        copy(pb, pa, cb[:b.nd], ca[:a.nd])
        copy(vb, va, cb[b.nd:], ca[a.nd:])
        copy(rb, ra, cb[b.nd:], ca[a.nd:])
        copy(ub, ua, list(b.input_names), list(a.input_names))
        return self.trajectory_return(nX, nU)

    tangent_trajectory_return = namedtuple("tangent_trajectory", "dX dU")

    def dproject(self, A, B, bdX, bdU, K):
        """Projection into the tangent trajectory space about a linearization (dsystem.py:460-471):
        dX[0] = bdX[0]; dU[k] = bdU[k] - K[k](dX[k] - bdX[k]); dX[k+1] = A[k] dX[k] + B[k] dU[k].
        One trajectory or a batch with a leading axis on every argument (a sequential recursion of
        matrix-vector products per rollout; evaluated on the host, vectorised over the batch)."""
        A, B, bdX, bdU, K = (np.asarray(x, float) for x in (A, B, bdX, bdU, K))
        dX, dU = np.zeros(bdX.shape), np.zeros(bdU.shape)
        dX[..., 0, :] = bdX[..., 0, :]
        for k in range(bdX.shape[-2] - 1):
            dU[..., k, :] = bdU[..., k, :] - np.einsum("...ij,...j->...i", K[..., k, :, :], dX[..., k, :] - bdX[..., k, :])
            dX[..., k + 1, :] = (np.einsum("...ij,...j->...i", A[..., k, :, :], dX[..., k, :])
                                 + np.einsum("...ij,...j->...i", B[..., k, :, :], dU[..., k, :]))
        return self.tangent_trajectory_return(dX, dU)

    # ---- f and the finite-difference self-checks (dsystem.py:253-281, 536-701) -------------------------
    error_return = namedtuple("derivative_error", "error exact_norm approx_norm")

    def f(self, X, U, k):
        """X[k+1] = f(X, U, k) for a batch of states / inputs at the time step k (DSystem.set + f,
        dsystem.py:229-281): X [n,nX], U [n,nU] -> [n,nX] = [q2; p2; (q2_kin - q1_kin)/dt]."""
        X, U = np.atleast_2d(np.asarray(X, float)), np.atleast_2d(np.asarray(U, float))
        t1, t2 = float(self._time[k]), float(self._time[k + 1])
        q1, p1, _ = self.split_state(X)
        u1, rho = self.split_input(U)
        out = self.varint.sys.step(q1, p1, t1, t2 - t1, nsteps=1, u1=u1[:, None, :] if self._nu else None,
                                   k2=rho[:, None, :] if self._nv else None, tolerance=self.varint.tolerance,
                                   params=self._rows(X.shape[0]))
        bad = np.flatnonzero(out["status"] != 0)
        if bad.size:
            raise ConvergenceError("%d of %d steps failed" % (bad.size, X.shape[0]), out["status"])
        v2 = (out["q2"][:, self._np:] - q1[:, self._np:]) / (t2 - t1)
        return self.build_state(out["q2"], out["p2"], v2)

    def _single_row(self):
        if self._params is not None and self._params[1].shape[0] != 1:
            raise ValueError("the check_* helpers need a single parameter row (set_parameters)")

    def _lin_at(self, X, U, k):
        self._single_row()
        n = X.shape[0]
        return self.linearize(X, U, np.full(n, self._time[k]), np.full(n, self._time[k + 1]))

    def _err(self, exact, approx):
        return self.error_return(float(np.linalg.norm(exact - approx)), float(np.linalg.norm(exact)),
                                 float(np.linalg.norm(approx)))

    def _perturbed(self, v, delta):
        """[2 n, n]: v + delta e_i (rows 0..n-1) and v - delta e_i (rows n..2n-1)."""
        n = v.shape[0]
        return np.concatenate([v[None] + delta * np.eye(n), v[None] - delta * np.eye(n)])

    def check_fdx(self, xk, uk, k, delta=1e-5):
        """f_dx against central differences of f (dsystem.py:536-562); the 2 nX perturbed states are
        one batch."""
        xk, uk = np.asarray(xk, float), np.asarray(uk, float)
        exact = self._lin_at(xk[None], uk[None], k).A[0]
        F = self.f(self._perturbed(xk, delta), np.tile(uk, (2 * self._nX, 1)), k)
        approx = ((F[:self._nX] - F[self._nX:]) / (2 * delta)).T
        return self._err(exact, approx)

    def check_fdu(self, xk, uk, k, delta=1e-5):
        """f_du against central differences of f (dsystem.py:565-591)."""
        xk, uk = np.asarray(xk, float), np.asarray(uk, float)
        exact = self._lin_at(xk[None], uk[None], k).B[0]
        F = self.f(np.tile(xk, (2 * self._nU, 1)), self._perturbed(uk, delta), k)
        approx = ((F[:self._nU] - F[self._nU:]) / (2 * delta)).T
        return self._err(exact, approx)

    def _second(self, xk, uk, k):
        """fdxdx(e_i), fdxdu(e_i), fdudu(e_i) for every unit vector e_i of the state space: one batch of nX
        instances of the z-contracted second-derivative kernel."""
        self._single_row()
        nX = self._nX
        t1, t2 = np.full(nX, self._time[k]), np.full(nX, self._time[k + 1])
        return self.second_derivatives(np.tile(xk, (nX, 1)), np.tile(uk, (nX, 1)), np.eye(nX), t1, t2)

    def check_fdxdx(self, xk, uk, k, delta=1e-5):
        """f_dxdx against central differences of f_dx (dsystem.py:594-625)."""
        xk, uk = np.asarray(xk, float), np.asarray(uk, float)
        exact = self._second(xk, uk, k)[0]                                   # [out i][a][b]
        A = self._lin_at(self._perturbed(xk, delta), np.tile(uk, (2 * self._nX, 1)), k).A
        approx = np.transpose((A[:self._nX] - A[self._nX:]) / (2 * delta), (1, 2, 0))   # [i][a][b = perturbed]
        return self._err(exact, approx)

    def check_fdxdu(self, xk, uk, k, delta=1e-5):
        """f_dxdu against central differences of f_dx (dsystem.py:628-660)."""
        xk, uk = np.asarray(xk, float), np.asarray(uk, float)
        exact = self._second(xk, uk, k)[1]                                   # [i][a][c]
        A = self._lin_at(np.tile(xk, (2 * self._nU, 1)), self._perturbed(uk, delta), k).A
        approx = np.transpose((A[:self._nU] - A[self._nU:]) / (2 * delta), (1, 2, 0))
        return self._err(exact, approx)

    def check_fdudu(self, xk, uk, k, delta=1e-5):
        """f_dudu against central differences of f_du (dsystem.py:663-701)."""
        xk, uk = np.asarray(xk, float), np.asarray(uk, float)
        exact = self._second(xk, uk, k)[2]                                   # [i][c][d]
        B = self._lin_at(np.tile(xk, (2 * self._nU, 1)), self._perturbed(uk, delta), k).B
        approx = np.transpose((B[:self._nU] - B[self._nU:]) / (2 * delta), (1, 2, 0))
        return self._err(exact, approx)

    # ---- the hot path ----------------------------------------------------------------------------------
    def linearize(self, X, U, t1, t2, X_hint=None, group=None, gather="nccl", everywhere=False):
        """A[i] = fdx, B[i] = fdu of instance i: DSystem.set(X[i], U[i], k, xk_hint=X_hint[i]) +
        fdx() + fdu() of the reference.  X [n,nX], U [n,nU], t1/t2 [n].

        group: a trep_b200.dist.Group (one process per GPU): the instances are block-partitioned over the
        ranks, every rank linearizes its block, and the A / B slabs are collected on rank 0 (every rank with
        everywhere=True) device to device: gather="nccl" (ncclSend/Recv or ncclAllGather on the finished
        slabs) or gather="peer" (rank 0's slab is mapped into every rank and the linearize kernel writes
        its block straight into it).  Ranks that do not receive the result return None."""
        return self._linearize(X, U, t1, t2, X_hint, group, gather, everywhere, 1)

    def _linearize(self, X, U, t1, t2, X_hint, group, gather, everywhere, per):
        """linearize, consecutive runs of `per` instances sharing a parameter row (the steps of one rollout)."""
        X, U = np.asarray(X, float), np.asarray(U, float)
        n = X.shape[0]
        world = 1 if group is None else group.world
        rank = 0 if group is None else group.rank
        lo, hi = shard_range(n, rank, world)
        q1, p1, _ = self.split_state(X[lo:hi])
        u1, rho2 = self.split_input(U[lo:hi])
        hint = None if X_hint is None else np.asarray(X_hint, float)[lo:hi, :self._np]
        t1 = np.broadcast_to(np.asarray(t1, float), (n,))[lo:hi]
        t2 = np.broadcast_to(np.asarray(t2, float), (n,))[lo:hi]
        params = self._rows(n, per)
        if params is not None:
            params = (params[0], np.ascontiguousarray(params[1][lo:hi]))
        if world == 1:
            out = self.varint.sys.linearize(q1, p1, u1, rho2, t1=t1, t2=t2, q2_guess=hint, tolerance=self.varint.tolerance,
                                            params=params)
            A, B, status = out["A"], out["B"], out["status"]
        else:
            A, B, status = self._linearize_sharded(q1, p1, u1, rho2, t1, t2, hint, n, lo, hi, group, gather, everywhere,
                                                   params)
            if A is None:
                return None
        bad = np.flatnonzero(status != 0)
        if bad.size:
            raise ConvergenceError("%d of %d linearizations failed (first: instance %d, status %d)"
                                   % (bad.size, n, bad[0], status[bad[0]]), status)
        return self.linearization_return(A, B)

    def _linearize_sharded(self, q1, p1, u1, rho2, t1, t2, hint, n, lo, hi, group, gather, everywhere, params=None):
        """This rank's block on its GPU, results collected on rank 0 without leaving device memory.  params: this
        block's parameter rows."""
        from . import dist, lib
        sys_, dev = self.varint.sys, self.varint.sys.device
        nX, nU, cnt = self._nX, self._nU, hi - lo
        up = lambda a: lib.DeviceBuffer(dev, a.shape, np.float64).upload(np.ascontiguousarray(a, dtype=np.float64))
        ins = dict(q1=up(q1), p1=up(p1), u1=up(u1) if self._nu else None, k2=up(rho2) if self._nv else None,
                   t1=up(t1), t2=up(t2), hint=None if hint is None else up(hint),
                   params=None if params is None else up(params[1]))
        dpar = None if params is None else (params[0], ins["params"])
        rowA, rowB = nX * nX * 8, nX * nU * 8
        root = group.rank == 0
        slabs = []
        try:
            if gather == "peer":
                # rank 0 owns [n] rows of A | B | status; every rank maps it and writes its own rows
                offB, offS = n * rowA, n * (rowA + rowB)
                slab = dist.SharedSlab(dev, group.exchange, n * (rowA + rowB + 4))
                slabs.append(slab)
                sys_.linearize_raw(True, cnt, ins["q1"], ins["p1"], ins["u1"], ins["k2"], slab.at(offS + lo * 4),
                                   t1=ins["t1"], t2=ins["t2"], q2_guess=ins["hint"], A=slab.at(lo * rowA),
                                   B=slab.at(offB + lo * rowB) if nU else None, tolerance=self.varint.tolerance,
                                   params=dpar)
                lib.synchronize(dev)
                group.barrier()          # every rank's stores have reached rank 0's HBM
                res = None
                if root:
                    raw = slab.local.download()
                    res = (raw[:offB].view(np.float64).reshape(n, nX, nX).copy(),
                           raw[offB:offS].view(np.float64).reshape(n, nX, nU).copy(),
                           raw[offS:offS + 4 * n].view(np.int32).copy())
                if everywhere:
                    raise ValueError('gather="peer" delivers to rank 0 only; use gather="nccl" with everywhere=True')
                group.barrier()          # nobody unmaps before rank 0 has read
                return res if root else (None, None, None)
            dA, dB = lib.DeviceBuffer(dev, (max(cnt, 1), nX, nX)), lib.DeviceBuffer(dev, (max(cnt, 1), nX, max(nU, 1)))
            dS = lib.DeviceBuffer(dev, (max(cnt, 1),), np.int32)
            slabs += [dA, dB, dS]
            sys_.linearize_raw(True, cnt, ins["q1"], ins["p1"], ins["u1"], ins["k2"], dS, t1=ins["t1"], t2=ins["t2"],
                               q2_guess=ins["hint"], A=dA, B=dB if nU else None, tolerance=self.varint.tolerance,
                               params=dpar)
            out = []
            for buf, rb, dt, shape in ((dA, rowA, np.float64, (n, nX, nX)), (dB, rowB, np.float64, (n, nX, nU)),
                                       (dS, 4, np.int32, (n,))):
                if rb == 0:
                    out.append(np.zeros(shape, dt))
                    continue
                full = dist.gather_rows(buf, cnt, n, rb, group.comm, dev, everywhere=everywhere)
                if full is None:
                    out.append(None)
                else:
                    out.append(full.download()[:n * rb].view(dt).reshape(shape).copy())
                    full.free()
            return tuple(out)
        finally:
            for b in list(ins.values()) + slabs:
                if b is not None:
                    (b.close if hasattr(b, "close") else b.free)()

    def second_derivatives(self, X, U, Z, t1, t2, X_hint=None):
        """z-contracted second derivatives of f for every instance: what the reference's
        fdxdx(z), fdxdu(z), fdudu(z) (dsystem.py:320-386) return after set(X[i], U[i], k).
        X [n,nX], U [n,nU], Z [n,nX], t1/t2 [n].  Returns (fdxdx [n,nX,nX], fdxdu [n,nX,nU],
        fdudu [n,nU,nU]); the full 30 tensors are never materialised."""
        return self._second_derivatives(X, U, Z, t1, t2, X_hint, 1)

    def _second_derivatives(self, X, U, Z, t1, t2, X_hint, per):
        """second_derivatives, consecutive runs of `per` instances sharing a parameter row (the steps of one rollout)."""
        X, U, Z = np.asarray(X, float), np.asarray(U, float), np.asarray(Z, float)
        n = X.shape[0]
        q1, p1, _ = self.split_state(X)
        u1, rho2 = self.split_input(U)
        hint = None if X_hint is None else np.asarray(X_hint, float)[:, :self._np]
        out = self.varint.sys.deriv2(q1, p1, u1, rho2, t1=np.broadcast_to(np.asarray(t1, float), (n,)),
                                     t2=np.broadcast_to(np.asarray(t2, float), (n,)), q2_guess=hint,
                                     tolerance=self.varint.tolerance, z=Z, tensors=False, params=self._rows(n, per))
        bad = np.flatnonzero(out["status"] != 0)
        if bad.size:
            raise ConvergenceError("%d of %d instances failed" % (bad.size, n), out["status"])
        return out["fdxdx"], out["fdxdu"], out["fdudu"]

    def calc_newton_model(self, X, U, A, B, K, l_dx, l_du, m_dx):
        """The dynamics' part of DOptimizer.calc_newton_model (doptimizer.py:319-345) for one trajectory or a
        batch of rollouts sharing `time`: the backward adjoint recursion
            z[n] = m_dx,   z[k] = l_dx[k] - l_du[k] K[k] + z[k+1] (A[k] - B[k] K[k])
        (n matrix-vector products per rollout, on the host) and then ONE launch of the z-contracted
        second-derivative kernel over every step of every rollout (step k contracts with z[k+1]).
        X [.., n+1, nX], U [.., n, nU], A / B / K per step, l_dx [.., n, nX], l_du [.., n, nU], m_dx [.., nX].
        Returns (z [.., n+1, nX], fdxdx [.., n, nX, nX], fdxdu [.., n, nX, nU], fdudu [.., n, nU, nU]): add the cost's
        own second derivatives to obtain Q(k), S(k), R(k)."""
        X, U = np.asarray(X, float), np.asarray(U, float)
        single = X.ndim == 2
        f = (lambda a: np.asarray(a, float)[None]) if single else (lambda a: np.asarray(a, float))
        X, U, A, B, K, l_dx, l_du, m_dx = (f(a) for a in (X, U, A, B, K, l_dx, l_du, m_dx))
        R, n = X.shape[0], X.shape[1] - 1
        Z = np.zeros((R, n + 1, self._nX))
        Z[:, n] = m_dx
        for k in reversed(range(n)):
            Acl = A[:, k] - np.einsum("rxu,ruy->rxy", B[:, k], K[:, k])
            Z[:, k] = l_dx[:, k] - np.einsum("ru,rux->rx", l_du[:, k], K[:, k]) + np.einsum("rx,rxy->ry", Z[:, k + 1], Acl)
        t1, t2 = np.tile(self._time[:n], R), np.tile(self._time[1:n + 1], R)
        xx, xu, uu = self._second_derivatives(X[:, :n].reshape(R * n, -1), U[:, :n].reshape(R * n, -1),
                                              Z[:, 1:].reshape(R * n, -1), t1, t2, X[:, 1:].reshape(R * n, -1), n)
        xx = xx.reshape(R, n, self._nX, self._nX); xu = xu.reshape(R, n, self._nX, self._nU)
        uu = uu.reshape(R, n, self._nU, self._nU)
        if single:
            return Z[0], xx[0], xu[0], uu[0]
        return Z, xx, xu, uu

    def linearize_trajectory(self, X, U, group=None, gather="nccl", everywhere=False):
        """Linearization about a trajectory (dsystem.py:406-423).  X [K+1, nX], U [K, nU] for one
        trajectory or X [R, K+1, nX], U [R, K, nU] for R rollouts sharing `time`.
        Returns (A, B) with shapes [..., K, nX, nX], [..., K, nX, nU] (None on the ranks of a `group` that
        do not receive the result, see linearize)."""
        X, U = np.asarray(X, float), np.asarray(U, float)
        single = X.ndim == 2
        if single:
            X, U = X[None], U[None]
        R, K = X.shape[0], X.shape[1] - 1
        assert U.shape[1] >= K and len(self._time) >= K + 1
        t1 = np.tile(self._time[:K], R)
        t2 = np.tile(self._time[1:K + 1], R)
        res = self._linearize(X[:, :K].reshape(R * K, -1), U[:, :K].reshape(R * K, -1), t1, t2,
                              X[:, 1:K + 1].reshape(R * K, -1), group, gather, everywhere, K)
        if res is None:
            return None
        A, B = res
        A = A.reshape(R, K, self._nX, self._nX)
        B = B.reshape(R, K, self._nX, self._nU)
        if single:
            A, B = A[0], B[0]
        return self.linearization_return(A, B)

    def _feedback_on_device(self, Xb, Ub, Q, R):
        """linearize -> Riccati sweep for Rn rollouts (Xb [Rn,K+1,nX], Ub [Rn,K,nU]), enqueued on the device without
        the A / B slabs leaving the GPU.  Q / R as calc_feedback_controller.  Returns a dict of device buffers:
        the linearization's inputs (q1, p1, u1, k2, hint, t1, t2, params), its outputs A, B, status, and the gains K
        with their status lqr_status; the caller synchronizes, calls _check_feedback and frees them (_free)."""
        from . import lib
        Rn, K = Xb.shape[0], Xb.shape[1] - 1
        Q = np.eye(self._nX) if Q is None else (np.stack([Q(k) for k in range(K + 1)]) if callable(Q) else np.asarray(Q, float))
        R = np.eye(self._nU) if R is None else (np.stack([R(k) for k in range(K)]) if callable(R) else np.asarray(R, float))
        sys_, dev = self.varint.sys, self.varint.sys.device
        nX, nU, nq, nd = self._nX, self._nU, self._nQ, self._np
        n = Rn * K
        up = lambda a, dt=np.float64: lib.DeviceBuffer(dev, a.shape, dt).upload(np.ascontiguousarray(a, dtype=dt))
        Xk = Xb[:, :K].reshape(n, nX)
        d = {}
        try:
            # inputs of the n = rollouts x steps independent linearizations, resident in HBM
            d["q1"], d["p1"] = up(Xk[:, :nq]), up(Xk[:, nq:nq + nd])
            d["u1"] = up(Ub[:, :K, :self._nu].reshape(n, -1)) if self._nu else None
            d["k2"] = up(Ub[:, :K, self._nu:].reshape(n, -1)) if self._nv else None
            d["hint"] = up(Xb[:, 1:K + 1, :nd].reshape(n, nd))
            d["t1"], d["t2"] = up(np.tile(self._time[:K], Rn)), up(np.tile(self._time[1:K + 1], Rn))
            d["A"], d["B"] = lib.DeviceBuffer(dev, (n, nX, nX)), lib.DeviceBuffer(dev, (n, nX, nU))
            d["status"] = lib.DeviceBuffer(dev, (n,), np.int32)
            d["Q"], d["R"] = up(Q), up(R)
            d["K"], d["lqr_status"] = lib.DeviceBuffer(dev, (Rn, K, nU, nX)), lib.DeviceBuffer(dev, (Rn,), np.int32)
            params = self._rows(n, K)
            d["params"] = None if params is None else up(params[1])
            d["refs"] = None if params is None else params[0]
            # linearize -> Riccati sweep without the A / B slabs leaving the GPU
            sys_.linearize_raw(True, n, d["q1"], d["p1"], d["u1"], d["k2"], d["status"], t1=d["t1"], t2=d["t2"],
                               q2_guess=d["hint"], A=d["A"], B=d["B"], tolerance=self.varint.tolerance,
                               params=self._dev_params(d))
            lib.lqr_raw(True, dev, Rn, K, nX, nU, d["A"], d["B"], d["Q"], d["R"], d["K"], d["lqr_status"],
                        q_per_step=Q.ndim == 3, r_per_step=R.ndim == 3)
        except BaseException:
            self._free(d)
            raise
        return d

    @staticmethod
    def _dev_params(d):
        return None if d["params"] is None else (d["refs"], d["params"])

    @staticmethod
    def _free(d):
        for b in d.values():
            if hasattr(b, "free"):
                b.free()

    @staticmethod
    def _check_feedback(d):
        """After a synchronize: raise ConvergenceError for a failed linearization or a singular Riccati step."""
        status, ls = d["status"].download(), d["lqr_status"].download()
        if np.any(status != 0):
            raise ConvergenceError("%d of %d linearizations failed" % (int(np.sum(status != 0)), status.size), status)
        if np.any(ls != 0):
            raise ConvergenceError("singular gamma in the Riccati sweep", ls)

    def calc_feedback_controller(self, X, U, Q=None, R=None, return_linearization=False):
        """DSystem.calc_feedback_controller (dsystem.py:474-494): linearize about (X, U), then the
        time-varying LQR gains (discopt.dlqr.solve_tv_lqr, dlqr.py:9-38) - both on the GPU, for one
        trajectory or a batch of rollouts.  Q / R: constant matrices or per-step stacks
        [K+1,nX,nX] / [K,nU,nU] (the reference takes functions Q(k), R(k)); identity by default."""
        from . import lib
        X, U = np.asarray(X, float), np.asarray(U, float)
        single = X.ndim == 2
        Xb, Ub = (X[None], U[None]) if single else (X, U)
        Rn, K = Xb.shape[0], Xb.shape[1] - 1
        nX, nU = self._nX, self._nU
        d = self._feedback_on_device(Xb, Ub, Q, R)
        try:
            lib.synchronize(self.varint.sys.device)
            self._check_feedback(d)
            Kfb = d["K"].download()
            A = d["A"].download().reshape(Rn, K, nX, nX) if return_linearization else None
            B = d["B"].download().reshape(Rn, K, nX, nU) if return_linearization else None
        finally:
            self._free(d)
        if single:
            Kfb = Kfb[0]
            A, B = (A[0], B[0]) if return_linearization else (None, None)
        if return_linearization:
            return Kfb, A, B
        return Kfb

    def calc_descent_direction(self, X, U, q, r, Q, S, R, Qproj=None, Rproj=None, newton=False, dx0=None,
                               return_linearization=False):
        """The descent direction of DOptimizer.calc_descent_direction (doptimizer.py:348-402) for one trajectory or
        R rollouts sharing `time`, as one chain of device launches:
            linearize -> LQR (Kproj, with Qproj / Rproj as calc_feedback_controller)
            [newton: adjoint sweep z (K = Kproj, l_dx = q[:K], l_du = r, m_dx = q[K]) -> z-contracted second
             derivatives, added to Q[:K] / S / R]
            -> LQ (trepb_lq_batch: K, C) -> tangent sweep dX[0] = dx0, dU[k] = -K[k] dX[k] - C[k],
               dX[k+1] = A[k] dX[k] + B[k] dU[k].
        q [K+1,nX], r [K,nU], Q [K+1,nX,nX], S [K,nX,nU] or None, R [K,nU,nU]: the LQ model (the cost's gradients
        and second derivatives along (X, U)), shared by the rollouts or one set per rollout (one more leading axis),
        as for lib.solve_tv_lq.  dx0: [nX] or [R,nX], default zero.  A, B, Kproj, K and C stay on the device; only
        (X, U), the cost terms and dx0 go in.  With newton=True the three z-contracted blocks are downloaded, added to
        Q / S / R on the host and uploaded again.
        Returns (Kproj, dX, dU), then z [..,K+1,nX] with newton=True, then A, B with return_linearization=True.
        With set_parameters, rollout r runs on row r in every launch."""
        from . import lib
        X, U = np.asarray(X, float), np.asarray(U, float)
        single = X.ndim == 2
        Xb, Ub = (X[None], U[None]) if single else (X, U)
        Rn, K = Xb.shape[0], Xb.shape[1] - 1
        nX, nU = self._nX, self._nU
        sys_, dev = self.varint.sys, self.varint.sys.device
        f = lambda a: None if a is None else np.asarray(a, float)
        q, r, Q, S, R = f(q), f(r), f(Q), f(S), f(R)
        # one cost per rollout when any term has the rollout axis, or when the Newton terms make it so
        per = newton or Q.ndim == 4 or q.ndim == 3 or r.ndim == 3 or R.ndim == 4 or (S is not None and S.ndim == 4)
        if per:
            roll = lambda a, sh: None if a is None else np.ascontiguousarray(np.broadcast_to(a, (Rn,) + sh))
            q, r, Q, R = roll(q, (K + 1, nX)), roll(r, (K, nU)), roll(Q, (K + 1, nX, nX)), roll(R, (K, nU, nU))
            S = roll(S, (K, nX, nU))
        up = lambda a: lib.DeviceBuffer(dev, a.shape, np.float64).upload(np.ascontiguousarray(a, dtype=np.float64))
        n = Rn * K
        d = self._feedback_on_device(Xb, Ub, Qproj, Rproj)
        try:
            z = None
            if newton:
                # costate on the device (step k's second derivatives contract with z[k+1] = z1[k]), then one launch
                # of the z-contracted second-derivative kernel over every step of every rollout
                d["l_dx"], d["l_du"], d["m_dx"] = up(q[:, :K]), up(r), up(q[:, K])
                d["z"], d["z1"] = lib.DeviceBuffer(dev, (Rn, K + 1, nX)), lib.DeviceBuffer(dev, (n, nX))
                lib.adjoint_raw(True, dev, Rn, K, nX, nU, d["A"], d["B"], d["m_dx"], d["z"], K=d["K"], l_dx=d["l_dx"],
                                l_du=d["l_du"], z1=d["z1"])
                d["fdxdx"], d["fdxdu"] = lib.DeviceBuffer(dev, (n, nX, nX)), lib.DeviceBuffer(dev, (n, nX, nU))
                d["fdudu"], d["d2_status"] = lib.DeviceBuffer(dev, (n, nU, nU)), lib.DeviceBuffer(dev, (n,), np.int32)
                sys_.deriv2_raw(True, n, d["q1"], d["p1"], d["u1"], d["k2"], d["d2_status"], {}, z=d["z1"],
                                fdxdx=d["fdxdx"], fdxdu=d["fdxdu"], fdudu=d["fdudu"], t1=d["t1"], t2=d["t2"],
                                q2_guess=d["hint"], tolerance=self.varint.tolerance, params=self._dev_params(d))
                lib.synchronize(dev)
                self._check_feedback(d)
                st = d["d2_status"].download()
                if np.any(st != 0):
                    raise ConvergenceError("%d of %d instances failed" % (int(np.sum(st != 0)), n), st)
                # the Newton terms are summed on the host (download, add, upload)
                Q = Q.copy()
                Q[:, :K] += d["fdxdx"].download().reshape(Rn, K, nX, nX)
                xu = d["fdxdu"].download().reshape(Rn, K, nX, nU)
                S = xu if S is None else S + xu
                R = R + d["fdudu"].download().reshape(Rn, K, nU, nU)
                z = d["z"].download()
            d["Qm"], d["Rm"], d["qm"], d["rm"] = up(Q), up(R), up(q), up(r)
            d["Sm"] = None if S is None else up(S)
            d["Klq"], d["C"] = lib.DeviceBuffer(dev, (Rn, K, nU, nX)), lib.DeviceBuffer(dev, (Rn, K, nU))
            d["lq_status"] = lib.DeviceBuffer(dev, (Rn,), np.int32)
            lib.lq_raw(True, dev, Rn, K, nX, nU, d["A"], d["B"], d["Qm"], d["Sm"], d["Rm"], d["qm"], d["rm"], d["Klq"],
                       d["C"], d["lq_status"], cost_per_rollout=per)
            # the tangent sweep runs with bdU = +C and x0 = -dx0: by linearity it returns exactly -dX, -dU (negation
            # is exact in floating point), which spares a device-side negation of C
            x0 = None
            if dx0 is not None:
                d["x0"] = x0 = up(-np.broadcast_to(np.asarray(dx0, float), (Rn, nX)))
            d["dX"], d["dU"] = lib.DeviceBuffer(dev, (Rn, K + 1, nX)), lib.DeviceBuffer(dev, (Rn, K, nU))
            lib.tangent_raw(True, dev, Rn, K, nX, nU, d["A"], d["B"], d["Klq"], d["dX"], d["dU"], bdU=d["C"], x0=x0)
            lib.synchronize(dev)
            self._check_feedback(d)
            ls = d["lq_status"].download()
            if np.any(ls != 0):
                raise ConvergenceError("singular gamma in the LQ solve", ls)
            out = [d["K"].download(), -d["dX"].download(), -d["dU"].download()]
            if newton:
                out.append(z)
            if return_linearization:
                out += [d["A"].download().reshape(Rn, K, nX, nX), d["B"].download().reshape(Rn, K, nX, nU)]
        finally:
            self._free(d)
        return tuple(o[0] for o in out) if single else tuple(out)

    def project(self, bX, bU, Kproj, use_hint=True):
        """DSystem.project (dsystem.py:426-457) for one candidate or a batch of candidates in one
        launch: X[0] = bX[0]; U[k] = bU[k] - Kproj[k] (X[k] - bX[k]); X[k+1] = f(X[k], U[k], k).
        bX [K+1,nX] / [R,K+1,nX], bU [K,nU] / [R,K,nU], Kproj [K,nU,nX] shared or [R,K,nU,nX].
        use_hint=False is DOptimizer.armijo_simulate's variant (no xk_hint, doptimizer.py:405-428): pass
        every Armijo step size's (X + lam dX, U + lam dU) as one batch.  Raises ConvergenceError with
        the per-candidate status / first failed step attached when a candidate fails (the reference
        returns the partial trajectory nX[:k], nU[:k] in that case)."""
        bX, bU = np.asarray(bX, float), np.asarray(bU, float)
        single = bX.ndim == 2
        if single:
            bX, bU = bX[None], bU[None]
        K = bX.shape[1] - 1
        if len(self._time) < K + 1:
            raise ValueError("the time base has %d points, the trajectory needs %d" % (len(self._time), K + 1))
        # the kernel steps on this system's own time grid, uniform or not (dsystem.py:426-457 uses self._time[k])
        out = self.varint.sys.project(bX, bU[:, :K], np.asarray(Kproj, float), self._time[0],
                                      float(self._time[1] - self._time[0]), use_hint=use_hint,
                                      tolerance=self.varint.tolerance, times=self._time[:K + 1],
                                      params=self._rows(bX.shape[0]))
        self.last_project = out
        bad = np.flatnonzero(out["status"] != 0)
        if bad.size:
            raise ConvergenceError("%d of %d closed-loop rollouts failed (first: candidate %d at step %d)"
                                   % (bad.size, bX.shape[0], bad[0], out["fail_step"][bad[0]]), out["status"])
        X, U = out["X"], out["U"]
        if single:
            X, U = X[0], U[0]
        return self.trajectory_return(X, U)

    def simulate(self, X0, U):
        """Rollouts X[k+1] = f(X[k], U[k], k) from X0 [R, nX] with U [R, K, nU] in one launch
        (what repeated DSystem.step calls do, dsystem.py:253-281).  Returns X [R, K+1, nX].  With set_parameters,
        rollout r runs on row r; the MidpointVI is left at the final states reached on those rows, while its own
        parameters (none) stay as they were."""
        X0, U = np.atleast_2d(np.asarray(X0, float)), np.asarray(U, float)
        if U.ndim == 2:
            U = U[None]
        R, K = U.shape[0], U.shape[1]
        if len(self._time) < K + 1:
            raise ValueError("the time base has %d points, the rollout needs %d" % (len(self._time), K + 1))
        dts = np.diff(self._time[:K + 1])
        q0, p0, _ = self.split_state(X0)
        u, rho = self.split_input(U)
        v = self.varint
        params = self._rows(X0.shape[0])   # rollout r on row r
        if params is not None and v._params is not None:
            raise ValueError("parameters are set on both the DSystem and its MidpointVI: clear one of them")
        v.initialize_from_state(self._time[0], q0, p0)
        out = v.simulate(K, float(dts[0]), u=u if self._nu else None, k=rho if self._nv else None, sample_every=1,
                         times=self._time[:K + 1], params=params)
        Q = np.concatenate([q0[:, None, :], out["traj_q"]], axis=1)
        P = np.concatenate([p0[:, None, :], out["traj_p"]], axis=1)
        X = np.zeros((R, K + 1, self._nX))
        X[..., :self._nQ] = Q
        X[..., self._nQ:self._nQ + self._np] = P
        if self._nv:
            X[:, 0, self._nQ + self._np:] = X0[:, self._nQ + self._np:]
            X[:, 1:, self._nQ + self._np:] = (Q[:, 1:, self._np:] - Q[:, :-1, self._np:]) / dts[None, :, None]
        return X
