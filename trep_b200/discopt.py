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

    def calc_stationary_controller(self, xk, uk, Q=None, R=None, k=0, S=None, tol=1e-13, max_iterations=64,
                                   return_linearization=False):
        """Stationary LQR about an equilibrium (no counterpart in the reference, whose dlqr is time-varying only):
        linearize at (xk, uk) over the time step time[k] -> time[k+1], then the stabilizing solution P of the discrete
        algebraic Riccati equation P = A^T P A - (A^T P B + S)(R + B^T P B)^-1 (B^T P A + S^T) + Q and the gain
        K = (R + B^T P B)^-1 (B^T P A + S^T), so that u = uk - K (x - xk) - both on the GPU, A / B never leaving it.
        xk [nX], uk [nU] for one equilibrium or [M,nX], [M,nU] for M of them; with set_parameters, model r runs on
        row r (one equilibrium with M parameter rows: that equilibrium under each of the M models).  Q [nX,nX] and
        R [nU,nU] (identity by default) and S [nX,nU] (None: zero) are shared by the models, or one per model with a
        leading axis.  Returns (K [..,nU,nX], P [..,nX,nX]) - without the leading axis for one equilibrium and at most
        one parameter row - and A, B as well with return_linearization=True.  Raises ConvergenceError with the
        per-model status when a linearization or a DARE solve fails (lib.DARE_* for the latter)."""
        from . import lib
        Xb, Ub, single = self._equilibria(xk, uk)
        n, nX, nU = Xb.shape[0], self._nX, self._nU
        Q = np.eye(nX) if Q is None else np.asarray(Q, float)
        R = np.eye(nU) if R is None else np.asarray(R, float)
        S = None if S is None else np.asarray(S, float)
        dev = self.varint.sys.device
        up = lambda a, dt=np.float64: lib.DeviceBuffer(dev, a.shape, dt).upload(np.ascontiguousarray(a, dtype=dt))
        d = {}
        try:
            self._linearize_equilibria(Xb, Ub, k, d)
            d["Q"], d["R"] = up(Q), up(R)
            d["S"] = None if S is None else up(S)
            d["K"], d["P"] = lib.DeviceBuffer(dev, (n, nU, nX)), lib.DeviceBuffer(dev, (n, nX, nX))
            d["dare_status"] = lib.DeviceBuffer(dev, (n,), np.int32)
            # linearize -> DARE without the A / B slabs leaving the GPU
            lib.dare_raw(True, dev, n, nX, nU, d["A"], d["B"], d["Q"], d["R"], d["dare_status"], K=d["K"], P=d["P"],
                         S=d["S"], q_per_rollout=Q.ndim == 3, r_per_rollout=R.ndim == 3,
                         s_per_rollout=S is not None and S.ndim == 3, tol=tol, max_iterations=max_iterations)
            lib.synchronize(dev)
            self._check_linearizations(d)
            ds = d["dare_status"].download()
            bad = np.flatnonzero(ds != lib.DARE_OK)
            if bad.size:
                raise ConvergenceError("the DARE solve failed for %d of %d models (first: model %d, %s)"
                                       % (bad.size, n, bad[0], lib.DARE_STATUS.get(int(ds[bad[0]]), "?")), ds)
            out = [d["K"].download(), d["P"].download()]
            if return_linearization:
                out += [d["A"].download(), d["B"].download()]
        finally:
            self._free(d)
        return tuple(o[0] for o in out) if single else tuple(out)

    def _equilibria(self, xk, uk):
        """(Xb [n,nX], Ub [n,nU], single) for calc_stationary_controller / evaluate_stationary_controller: one
        equilibrium with M parameter rows is repeated M times; single = one equilibrium and at most one row."""
        xk, uk = np.asarray(xk, float), np.asarray(uk, float)
        single = xk.ndim == 1
        Xb, Ub = np.atleast_2d(xk), np.atleast_2d(uk)
        rows = 1 if self._params is None else self._params[1].shape[0]
        if Xb.shape[0] == 1 and rows > 1:
            Xb, Ub, single = np.repeat(Xb, rows, axis=0), np.repeat(Ub, rows, axis=0), False
        if Ub.shape[0] != Xb.shape[0]:
            raise ValueError("xk has %d equilibria, uk %d" % (Xb.shape[0], Ub.shape[0]))
        return Xb, Ub, single

    def _linearize_equilibria(self, Xb, Ub, k, d):
        """Launch the linearization at the equilibria (Xb, Ub) over time[k] -> time[k+1], model r on parameter row r:
        A / B / status into d["A"], d["B"], d["status"] on the device (no synchronize; see _check_linearizations)."""
        from . import lib
        n, nX, nU, nq, nd = Xb.shape[0], self._nX, self._nU, self._nQ, self._np
        sys_, dev = self.varint.sys, self.varint.sys.device
        up = lambda a, dt=np.float64: lib.DeviceBuffer(dev, a.shape, dt).upload(np.ascontiguousarray(a, dtype=dt))
        d["q1"], d["p1"] = up(Xb[:, :nq]), up(Xb[:, nq:nq + nd])
        d["u1"] = up(Ub[:, :self._nu]) if self._nu else None
        d["k2"] = up(Ub[:, self._nu:]) if self._nv else None
        d["hint"] = up(Xb[:, :nd])                     # at an equilibrium the dynamic configs stay where they are
        d["t1"], d["t2"] = up(np.full(n, self._time[k])), up(np.full(n, self._time[k + 1]))
        d["A"], d["B"] = lib.DeviceBuffer(dev, (n, nX, nX)), lib.DeviceBuffer(dev, (n, nX, nU))
        d["status"] = lib.DeviceBuffer(dev, (n,), np.int32)
        params = self._rows(n)
        d["params"] = None if params is None else up(params[1])
        d["refs"] = None if params is None else params[0]
        sys_.linearize_raw(True, n, d["q1"], d["p1"], d["u1"], d["k2"], d["status"], t1=d["t1"], t2=d["t2"],
                           q2_guess=d["hint"], A=d["A"], B=d["B"], tolerance=self.varint.tolerance,
                           params=self._dev_params(d))

    @staticmethod
    def _check_linearizations(d):
        """After a synchronize: raise ConvergenceError for a failed linearization of _linearize_equilibria."""
        status = d["status"].download()
        if np.any(status != 0):
            raise ConvergenceError("%d of %d linearizations failed" % (int(np.sum(status != 0)), status.size), status)

    def evaluate_stationary_controller(self, xk, uk, K, Q=None, R=None, k=0, S=None, x0=None, cross=True,
                                       return_P=False, tol=1e-13, max_iterations=64):
        """Closed-loop stability and infinite-horizon cost of stationary gains under every model (no counterpart in
        the reference): linearize at the equilibrium (xk, uk) exactly as calc_stationary_controller does (model m on
        parameter row m), then for each gain K_g and model m the solution P of the discrete Lyapunov equation
        P = A_c^T P A_c + Q_c, A_c = A_m - B_m K_g, Q_c = Q - S K_g - K_g^T S^T + K_g^T R K_g (the cost-to-go of
        u = uk - K_g (x - xk) under the stage cost dx^T Q dx + 2 dx^T S du + du^T R du), on the GPU with A / B never
        leaving it.  K [nU,nX] or [G,nU,nX]; Q / R / S as for calc_stationary_controller.  cost = x0^T P x0 for the
        initial deviation x0 [nX], or trace(P) without it (the expected cost from x0 ~ N(0, I)); +inf where the
        closed loop is not certified stable.  cross=True evaluates every gain under every model: returns
        (cost [G,M], status [G,M]); cross=False gain m under model m only (G = M): (cost [M], status [M]).  Without the
        G axis for K [nU,nX], without the M axis for one equilibrium and at most one parameter row.  status is
        lib.DLYAP_STABLE (0) exactly when the doubling certified rho(A_c) < 1, else lib.DLYAP_NOT_CONVERGED /
        lib.DLYAP_NONFINITE.  With return_P=True P [.., nX, nX] comes third.  Raises ConvergenceError when a
        linearization fails."""
        from . import lib
        Xb, Ub, single = self._equilibria(xk, uk)
        M, nX, nU = Xb.shape[0], self._nX, self._nU
        K = np.asarray(K, float)
        one_gain = K.ndim == 2
        Kb = np.ascontiguousarray(K[None] if one_gain else K)
        if Kb.ndim != 3 or Kb.shape[1:] != (nU, nX):
            raise ValueError("K must be [%d,%d] or [G,%d,%d]" % (nU, nX, nU, nX))
        G = Kb.shape[0]
        if not cross and not one_gain and G != M:
            raise ValueError("cross=False pairs gain m with model m: %d gains, %d models" % (G, M))
        Q = np.eye(nX) if Q is None else np.asarray(Q, float)
        R = np.eye(nU) if R is None else np.asarray(R, float)
        S = None if S is None else np.asarray(S, float)
        if cross:
            gi, mi = np.repeat(np.arange(G), M), np.tile(np.arange(M), G)
        else:
            gi, mi = np.zeros(M, int) if one_gain else np.arange(M), np.arange(M)
        pairs = gi.size
        dev = self.varint.sys.device
        up = lambda a, dt=np.float64: lib.DeviceBuffer(dev, a.shape, dt).upload(np.ascontiguousarray(a, dtype=dt))
        d = {}
        try:
            self._linearize_equilibria(Xb, Ub, k, d)
            d["K"], d["Q"], d["R"] = up(Kb), up(Q), up(R)
            d["S"] = None if S is None else up(S)
            d["gi"], d["mi"] = up(gi, np.int32), up(mi, np.int32)
            if x0 is None:
                d["x0"], d["W"] = None, up(np.eye(nX))
            else:
                d["x0"], d["W"] = up(np.asarray(x0, float).reshape(nX)), None
            d["cost"] = lib.DeviceBuffer(dev, (pairs,))
            d["P"] = lib.DeviceBuffer(dev, (pairs, nX, nX)) if return_P else None
            d["dlyap_status"] = lib.DeviceBuffer(dev, (pairs,), np.int32)
            # linearize -> Lyapunov without the A / B slabs leaving the GPU
            lib.dlyap_raw(True, dev, pairs, G, M, nX, nU, d["A"], d["B"], d["K"], d["Q"], d["R"], d["dlyap_status"],
                          S=d["S"], gain_index=d["gi"], model_index=d["mi"], x0=d["x0"], W=d["W"], P=d["P"],
                          cost=d["cost"], q_per_model=Q.ndim == 3, r_per_model=R.ndim == 3,
                          s_per_model=S is not None and S.ndim == 3, tol=tol, max_iterations=max_iterations)
            lib.synchronize(dev)
            self._check_linearizations(d)
            out = [d["cost"].download(), d["dlyap_status"].download()]
            if return_P:
                out.append(d["P"].download())
        finally:
            self._free(d)
        lead = (G, M) if cross else (M,)
        out = [o.reshape(lead + o.shape[1:]) for o in out]
        if cross and one_gain:
            out, lead = [o[0] for o in out], (M,)
        if single:
            out = [np.take(o, 0, axis=len(lead) - 1) for o in out]
        return tuple(out)

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
        Q / S / R on the host and uploaded again (discopt.DOptimizer builds its model on the device instead).
        Returns (Kproj, dX, dU), then z [..,K+1,nX] with newton=True, then A, B with return_linearization=True.
        With set_parameters, rollout r runs on row r in every launch."""
        X, U = np.asarray(X, float), np.asarray(U, float)
        single = X.ndim == 2
        Xb, Ub = (X[None], U[None]) if single else (X, U)
        Rn, K = Xb.shape[0], Xb.shape[1] - 1
        nX, nU = self._nX, self._nU
        d = self._descent_on_device(Xb, Ub, Qproj, Rproj, newton, dx0, _HostModel(self, Rn, K, newton, q, r, Q, S, R))
        try:
            out = [d["K"].download(), -d["dX"].download(), -d["dU"].download()]
            if newton:
                out.append(d["z"].download())
            if return_linearization:
                out += [d["A"].download().reshape(Rn, K, nX, nX), d["B"].download().reshape(Rn, K, nX, nU)]
        finally:
            self._free(d)
        return tuple(o[0] for o in out) if single else tuple(out)

    def _descent_on_device(self, Xb, Ub, Qproj, Rproj, newton, dx0, model):
        """The device chain of calc_descent_direction for Rn rollouts (Xb [Rn,K+1,nX], Ub [Rn,K,nU]):
            linearize -> LQR (Kproj) -> model.gradients [-> adjoint -> deriv2] -> model.hessians -> LQ -> tangent sweep.
        `model` supplies the LQ model: gradients(d) puts q / r in d["qm"] / d["rm"] (and, for the adjoint, l_dx / m_dx in
        d["l_dx"] / d["m_dx"]); hessians(d, newton) puts Q / S / R in d["Qm"] / d["Sm"] / d["Rm"], adding the z-contracted
        blocks d["fdxdx"], d["fdxdu"], d["fdudu"] with newton=True, and returns cost_per_rollout.  Synchronizes and
        raises ConvergenceError on a failed launch; otherwise returns the dict of device buffers (the caller frees it
        with _free), whose d["dX"] / d["dU"] hold -dX / -dU (see below) and d["K"] the gains Kproj."""
        from . import lib
        Rn, K = Xb.shape[0], Xb.shape[1] - 1
        nX, nU = self._nX, self._nU
        sys_, dev = self.varint.sys, self.varint.sys.device
        up = lambda a: lib.DeviceBuffer(dev, a.shape, np.float64).upload(np.ascontiguousarray(a, dtype=np.float64))
        n = Rn * K
        d = self._feedback_on_device(Xb, Ub, Qproj, Rproj)
        try:
            model.gradients(d)
            if newton:
                # costate on the device (step k's second derivatives contract with z[k+1] = z1[k]), then one launch
                # of the z-contracted second-derivative kernel over every step of every rollout
                d["z"], d["z1"] = lib.DeviceBuffer(dev, (Rn, K + 1, nX)), lib.DeviceBuffer(dev, (n, nX))
                lib.adjoint_raw(True, dev, Rn, K, nX, nU, d["A"], d["B"], d["m_dx"], d["z"], K=d["K"], l_dx=d["l_dx"],
                                l_du=d["rm"], z1=d["z1"])
                d["fdxdx"], d["fdxdu"] = lib.DeviceBuffer(dev, (n, nX, nX)), lib.DeviceBuffer(dev, (n, nX, nU))
                d["fdudu"], d["d2_status"] = lib.DeviceBuffer(dev, (n, nU, nU)), lib.DeviceBuffer(dev, (n,), np.int32)
                sys_.deriv2_raw(True, n, d["q1"], d["p1"], d["u1"], d["k2"], d["d2_status"], {}, z=d["z1"],
                                fdxdx=d["fdxdx"], fdxdu=d["fdxdu"], fdudu=d["fdudu"], t1=d["t1"], t2=d["t2"],
                                q2_guess=d["hint"], tolerance=self.varint.tolerance, params=self._dev_params(d))
            per = model.hessians(d, newton)
            d["Klq"], d["C"] = lib.DeviceBuffer(dev, (Rn, K, nU, nX)), lib.DeviceBuffer(dev, (Rn, K, nU))
            d["lq_status"] = lib.DeviceBuffer(dev, (Rn,), np.int32)
            lib.lq_raw(True, dev, Rn, K, nX, nU, d["A"], d["B"], d["Qm"], d.get("Sm"), d["Rm"], d["qm"], d["rm"],
                       d["Klq"], d["C"], d["lq_status"], cost_per_rollout=per)
            # the tangent sweep runs with bdU = +C and x0 = -dx0: by linearity it returns exactly -dX, -dU (negation
            # is exact in floating point), which spares a device-side negation of C
            x0 = None
            if dx0 is not None:
                d["x0"] = x0 = up(-np.broadcast_to(np.asarray(dx0, float), (Rn, nX)))
            d["dX"], d["dU"] = lib.DeviceBuffer(dev, (Rn, K + 1, nX)), lib.DeviceBuffer(dev, (Rn, K, nU))
            lib.tangent_raw(True, dev, Rn, K, nX, nU, d["A"], d["B"], d["Klq"], d["dX"], d["dU"], bdU=d["C"], x0=x0)
            lib.synchronize(dev)
            self._check_feedback(d)
            if newton:
                self._check_d2(d, n)
            ls = d["lq_status"].download()
            if np.any(ls != 0):
                raise ConvergenceError("singular gamma in the LQ solve", ls)
        except BaseException:
            self._free(d)
            raise
        return d

    @staticmethod
    def _check_d2(d, n):
        st = d["d2_status"].download()
        if np.any(st != 0):
            raise ConvergenceError("%d of %d instances failed" % (int(np.sum(st != 0)), n), st)

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


class _HostModel:
    """The LQ model of DSystem.calc_descent_direction given as host arrays: uploaded as they are, and with newton=True
    the z-contracted blocks are downloaded, summed into Q / S / R on the host and uploaded again."""

    def __init__(self, dsys, Rn, K, newton, q, r, Q, S, R):
        f = lambda a: None if a is None else np.asarray(a, float)
        q, r, Q, S, R = f(q), f(r), f(Q), f(S), f(R)
        nX, nU = dsys.nX, dsys.nU
        # one cost per rollout when any term has the rollout axis, or when the Newton terms make it so
        self.per = newton or Q.ndim == 4 or q.ndim == 3 or r.ndim == 3 or R.ndim == 4 or (S is not None and S.ndim == 4)
        if self.per:
            roll = lambda a, sh: None if a is None else np.ascontiguousarray(np.broadcast_to(a, (Rn,) + sh))
            q, r, Q, R = roll(q, (K + 1, nX)), roll(r, (K, nU)), roll(Q, (K + 1, nX, nX)), roll(R, (K, nU, nU))
            S = roll(S, (K, nX, nU))
        self.dsys, self.Rn, self.K, self.q, self.r, self.Q, self.S, self.R = dsys, Rn, K, q, r, Q, S, R

    def _up(self, a):
        from . import lib
        return lib.DeviceBuffer(self.dsys.varint.sys.device, a.shape, np.float64).upload(np.ascontiguousarray(a))

    def gradients(self, d):
        d["qm"], d["rm"] = self._up(self.q), self._up(self.r)
        if self.per:
            d["l_dx"], d["m_dx"] = self._up(self.q[:, :self.K]), self._up(self.q[:, self.K])

    def hessians(self, d, newton):
        from . import lib
        Q, S, R, Rn, K, ds = self.Q, self.S, self.R, self.Rn, self.K, self.dsys
        if newton:
            lib.synchronize(ds.varint.sys.device)
            ds._check_feedback(d)
            ds._check_d2(d, Rn * K)
            # the Newton terms are summed on the host (download, add, upload)
            nX, nU = ds.nX, ds.nU
            Q = Q.copy()
            Q[:, :K] += d["fdxdx"].download().reshape(Rn, K, nX, nX)
            xu = d["fdxdu"].download().reshape(Rn, K, nX, nU)
            S = xu if S is None else S + xu
            R = R + d["fdudu"].download().reshape(Rn, K, nU, nU)
        d["Qm"], d["Rm"] = self._up(Q), self._up(R)
        d["Sm"] = None if S is None else self._up(S)
        return self.per


# ---- the tracking cost and the batched optimiser -------------------------------------------------------------------
class DCost:
    """The quadratic tracking cost of trep.discopt.DCost (dcost.py):
        l(x, u, k) = (dx^T Q dx + du^T R du) / 2,  m(x) = dx_K^T Q dx_K / 2,  dx = x - xd[k],  du = u - ud[k].
    xd [K+1,nX] and ud [K,nU] are one reference, or [R,K+1,nX] / [R,K,nU] one per rollout.  The methods take one state
    / input, or one per rollout with a leading axis; DOptimizer evaluates the same cost on the GPU
    (lib.track_cost)."""

    def __init__(self, xd, ud, Q, R):
        self.xd, self.ud = np.array(xd, dtype=float), np.array(ud, dtype=float)
        self.Q, self.R = np.array(Q, dtype=float), np.array(R, dtype=float)

    @property
    def per_rollout(self):
        return self.xd.ndim == 3

    def l(self, xk, uk, k):
        dx, du = np.asarray(xk, float) - self.xd[..., k, :], np.asarray(uk, float) - self.ud[..., k, :]
        return 0.5 * (np.sum(dx * (dx @ self.Q.T), axis=-1) + np.sum(du * (du @ self.R.T), axis=-1))

    def m(self, xf):
        dx = np.asarray(xf, float) - self.xd[..., -1, :]
        return 0.5 * np.sum(dx * (dx @ self.Q.T), axis=-1)

    def l_dx(self, xk, uk, k):
        return (np.asarray(xk, float) - self.xd[..., k, :]) @ self.Q

    def l_du(self, xk, uk, k):
        return (np.asarray(uk, float) - self.ud[..., k, :]) @ self.R

    def m_dx(self, xf):
        return (np.asarray(xf, float) - self.xd[..., -1, :]) @ self.Q

    def l_dxdx(self, xk, uk, k):
        return self.Q

    def l_dudu(self, xk, uk, k):
        return self.R

    def l_dxdu(self, xk, uk, k):
        return np.zeros((self.Q.shape[0], self.R.shape[0]))

    def m_dxdx(self, xf):
        return self.Q


STEP_ACCEPTED = 0       # a step size passed the Armijo test (DOptimizer.last_status)
STEP_CONVERGED = 1      # |dcost| < descent_tolerance
ARMIJO_FAILED = -1      # no step size passed within armijo_max_iterations; the trajectory was kept


class _TrackModel:
    """The LQ model of a DOptimizer step built on the device by the track kernel (trepb_track_batch_dev): q / r /
    l_dx / m_dx and cost0 from the DCost along (X, U), then Q / S / R per rollout in the layout the LQ solve reads:
    identity weights for "steepest", the DCost weights for "quasi", and for "newton" those plus the z-contracted
    blocks, each sum one IEEE addition."""

    def __init__(self, opt, Xb, Ub, ref_rows, method):
        self.opt, self.Xb, self.Ub, self.ref_rows, self.method = opt, Xb, Ub, ref_rows, method

    def gradients(self, d):
        from . import lib
        opt = self.opt
        ds, dev = opt.dsys, opt.dsys.varint.sys.device
        Rn, K = self.Xb.shape[0], self.Xb.shape[1] - 1
        nX, nU = ds.nX, ds.nU
        opt._upload_cost(d, self.Xb, self.Ub, self.ref_rows)
        d["qm"], d["rm"] = lib.DeviceBuffer(dev, (Rn, K + 1, nX)), lib.DeviceBuffer(dev, (Rn, K, nU))
        d["l_dx"], d["m_dx"] = lib.DeviceBuffer(dev, (Rn, K, nX)), lib.DeviceBuffer(dev, (Rn, nX))
        d["cost"] = lib.DeviceBuffer(dev, (Rn,))
        model = {}
        if self.method == "quasi":
            d["Qm"], d["Rm"] = lib.DeviceBuffer(dev, (Rn, K + 1, nX, nX)), lib.DeviceBuffer(dev, (Rn, K, nU, nU))
            model = dict(Qm=d["Qm"], Rm=d["Rm"])
        lib.track_raw(True, dev, Rn, K, nX, nU, nref=d["nref"], X=d["X"], U=d["U"], Xd=d["Xd"], Ud=d["Ud"], Q=d["Qc"],
                      R=d["Rc"], ref_index=d.get("ref_index"), q=d["qm"], r=d["rm"], l_dx=d["l_dx"], m_dx=d["m_dx"],
                      cost=d["cost"], **model)

    def hessians(self, d, newton):
        from . import lib
        if self.method == "quasi":
            return True
        ds, dev = self.opt.dsys, self.opt.dsys.varint.sys.device
        Rn, K = self.Xb.shape[0], self.Xb.shape[1] - 1
        nX, nU = ds.nX, ds.nU
        d["Qm"], d["Rm"] = lib.DeviceBuffer(dev, (Rn, K + 1, nX, nX)), lib.DeviceBuffer(dev, (Rn, K, nU, nU))
        if newton:
            d["Sm"] = lib.DeviceBuffer(dev, (Rn, K, nX, nU))
            lib.track_raw(True, dev, Rn, K, nX, nU, Q=d["Qc"], R=d["Rc"], fdxdx=d["fdxdx"], fdxdu=d["fdxdu"],
                          fdudu=d["fdudu"], Qm=d["Qm"], Sm=d["Sm"], Rm=d["Rm"])
        else:   # steepest: Q = I, R = I, S = 0
            up = lambda a: lib.DeviceBuffer(dev, a.shape).upload(a)
            d["I_x"], d["I_u"] = up(np.eye(nX)), up(np.eye(nU))
            lib.track_raw(True, dev, Rn, K, nX, nU, Q=d["I_x"], R=d["I_u"], Qm=d["Qm"], Rm=d["Rm"])
        return True


class DOptimizer:
    """A batched trep.discopt.DOptimizer (doptimizer.py) for a DCost: R independent trajectory-optimisation problems
    (multi-start guesses, or plausible models through DSystem.set_parameters) per launch.  Every method takes one
    trajectory (X [K+1,nX], U [K,nU]) or R rollouts with a leading axis.  The cost, its gradient, the LQ model with
    the Newton terms, the Armijo candidates and their costs stay on the GPU; the host sees the costs, the statuses and
    the accepted trajectories.

    The defaults are believed to be the reference's (beta 0.7, alpha 1e-5, 30 Armijo iterations, descent tolerance
    1e-6, 10 first-method iterations, "quasi" then "newton"); they were not checked against its source.
    optimize_ic=True (a solve against P(0) inside the chain) and monitors are not supported."""
    descent_return = namedtuple("descent", "Kproj dX dU")
    armijo_search_return = namedtuple("armijo_search", "nX nU cost")
    step_return = namedtuple("step", "converged X U dcost cost")

    def __init__(self, dsys, cost, first_method_iterations=10, armijo_batch=8):
        self.dsys, self.cost = dsys, cost
        self.optimize_ic = False
        self.Qproj = self.Rproj = None
        self.armijo_beta = 0.7
        self.armijo_alpha = 0.00001
        self.armijo_max_iterations = 30
        self.descent_tolerance = 1e-6
        self.first_method_iterations = first_method_iterations
        self.first_method = "quasi"
        self.second_method = "newton"
        self.armijo_batch = armijo_batch
        self.last_status = None        # per rollout, after step / armijo_search / optimize
        self.last_armijo_m = None      # per rollout: the accepted m of the last search, -1 if none

    # ---- helpers -----------------------------------------------------------------------------------------------
    def _batch(self, X, U):
        X, U = np.asarray(X, float), np.asarray(U, float)
        single = X.ndim == 2
        return single, np.ascontiguousarray(X[None] if single else X), np.ascontiguousarray(U[None] if single else U)

    def _ref_rows(self, rows):
        """ref_index of the trajectories of rollouts `rows` (None: every rollout tracks the one reference)."""
        return np.asarray(rows, np.int32) if self.cost.per_rollout else None

    def _upload_cost(self, d, Xb, Ub, ref_rows):
        """X, U, the references, the weights and the reference index on the device, in d."""
        from . import lib
        dev = self.dsys.varint.sys.device
        up = lambda a, dt=np.float64: lib.DeviceBuffer(dev, np.shape(a), dt).upload(np.ascontiguousarray(a, dtype=dt))
        K = Xb.shape[1] - 1
        xd = self.cost.xd if self.cost.per_rollout else self.cost.xd[None]
        ud = self.cost.ud if self.cost.per_rollout else self.cost.ud[None]
        if xd.shape[1] < K + 1 or ud.shape[1] < K:
            raise ValueError("the reference has %d states, the trajectory %d" % (xd.shape[1], K + 1))
        d["X"], d["U"] = up(Xb), up(Ub)
        d["Xd"], d["Ud"] = up(xd[:, :K + 1]), up(ud[:, :K])
        d["Qc"], d["Rc"] = up(self.cost.Q), up(self.cost.R)
        d["nref"] = xd.shape[0]
        d["ref_index"] = None if ref_rows is None else up(ref_rows, np.int32)

    def _costs(self, Xb, Ub, dX=None, dU=None):
        from . import lib
        rows = self._ref_rows(np.arange(Xb.shape[0]))
        K = Xb.shape[1] - 1
        xd, ud = self.cost.xd[..., :K + 1, :], self.cost.ud[..., :K, :]
        return lib.track_cost(Xb, Ub, xd, ud, self.cost.Q, self.cost.R, ref_index=rows, dX=dX, dU=dU,
                              outputs=("cost", "dcost") if dX is not None else ("cost",),
                              device=self.dsys.varint.sys.device)

    def _params_for(self, rows):
        """DSystem parameters restricted to rollouts `rows` (None when they are not per rollout)."""
        p = self.dsys._params
        if p is None or p[1].shape[0] == 1:
            return None
        return p[0], np.ascontiguousarray(p[1][rows])

    # ---- the reference's interface -------------------------------------------------------------------------------
    def calc_cost(self, X, U):
        """DOptimizer.calc_cost: sum_k l(X[k], U[k], k) + m(X[K]), on the GPU."""
        single, Xb, Ub = self._batch(X, U)
        c = self._costs(Xb, Ub)["cost"]
        return float(c[0]) if single else c

    def calc_dcost(self, X, U, dX, dU):
        """DOptimizer.calc_dcost: sum_k l_dx . dX[k] + l_du . dU[k] + m_dx . dX[K], on the GPU."""
        single, Xb, Ub = self._batch(X, U)
        _, dXb, dUb = self._batch(dX, dU)
        c = self._costs(Xb, Ub, dXb, dUb)["dcost"]
        return float(c[0]) if single else c

    def _direction(self, Xb, Ub, rows, method):
        """The device chain of one descent direction for rollouts `rows`; returns its buffers (caller frees)."""
        if self.optimize_ic:
            raise ValueError("optimize_ic=True is not supported")
        if method not in ("steepest", "quasi", "newton"):
            raise ValueError("Invalid descent direction method: %r" % (method,))
        ds = self.dsys
        saved = ds._params
        sub = self._params_for(rows)
        if sub is not None:
            ds._params = sub
        try:
            return ds._descent_on_device(Xb, Ub, self.Qproj, self.Rproj, method == "newton", None,
                                         _TrackModel(self, Xb, Ub, self._ref_rows(rows), method))
        finally:
            ds._params = saved

    def calc_descent_direction(self, X, U, method="steepest"):
        """DOptimizer.calc_descent_direction: (Kproj, dX, dU).  The model (Q, R, S) stays on the device and is not
        returned."""
        single, Xb, Ub = self._batch(X, U)
        d = self._direction(Xb, Ub, np.arange(Xb.shape[0]), method)
        try:
            out = (d["K"].download(), -d["dX"].download(), -d["dU"].download())
        finally:
            self.dsys._free(d)
        return self.descent_return(*(o[0] for o in out)) if single else self.descent_return(*out)

    def _dcost_on_device(self, d, Rn, K):
        """dcost0 of the chain's direction: the track kernel on d["dX"] / d["dU"], which hold -dX / -dU (every
        product and sum is then exactly negated)."""
        from . import lib
        dev = self.dsys.varint.sys.device
        d["dcost"] = lib.DeviceBuffer(dev, (Rn,))
        lib.track_raw(True, dev, Rn, K, self.dsys.nX, self.dsys.nU, nref=d["nref"], X=d["X"], U=d["U"], Xd=d["Xd"],
                      Ud=d["Ud"], Q=d["Qc"], R=d["Rc"], ref_index=d.get("ref_index"), dX=d["dX"], dU=d["dU"],
                      dcost=d["dcost"])
        return -d["dcost"].download()

    def _search(self, d, Xb, Ub, rows, active, cost0, dcost0):
        """Armijo search of DOptimizer.armijo_search for the rollouts at positions `active` of this batch (rows: their
        rollout indices in the problem), on the buffers d holds: X, U, Xd, Ud, Qc, Rc, ref_index, dX / dU (= -dX /
        -dU) and K (Kproj).  Step sizes beta^m in batches of armijo_batch: one candidates launch, one project launch
        over the searching rollouts x M and one track launch for the candidates' costs; each rollout accepts the first
        m with cost1 < cost0 + alpha beta^m dcost0.  Returns (X, U, cost, status, m)."""
        from . import lib
        ds = self.dsys
        sys_, dev = ds.varint.sys, ds.varint.sys.device
        Rn, K = Xb.shape[0], Xb.shape[1] - 1
        nX, nU = ds.nX, ds.nU
        Xn, Un, cost = Xb.copy(), Ub.copy(), np.array(cost0, float)
        status = np.zeros(Rn, np.int32)
        macc = np.full(Rn, -1)
        up = lambda a, dt=np.float64: lib.DeviceBuffer(dev, np.shape(a), dt).upload(np.ascontiguousarray(a, dtype=dt))
        times = up(ds.time[:K + 1])
        par = ds._params
        try:
            g = np.asarray(active, dtype=np.int64)
            m0 = 0
            while g.size and m0 < self.armijo_max_iterations:
                ms = list(range(m0, min(m0 + self.armijo_batch, self.armijo_max_iterations)))
                lam = np.array([self.armijo_beta ** m for m in ms])
                M, G = len(ms), g.size
                n = G * M
                b = {}
                try:
                    b["rows"] = None if G == Rn else up(g, np.int32)
                    b["lam"] = up(-lam)   # -lam times -dX is exactly lam dX
                    b["bX"], b["bU"] = lib.DeviceBuffer(dev, (n, K + 1, nX)), lib.DeviceBuffer(dev, (n, K, nU))
                    b["Kc"] = lib.DeviceBuffer(dev, (n, K, nU, nX))
                    lib.candidates_raw(True, dev, G, M, K, nX, nU, b["lam"], d["X"], d["U"], d["dX"], d["dU"], d["K"],
                                       b["bX"], b["bU"], b["Kc"], rows=b["rows"])
                    b["pX"], b["pU"] = lib.DeviceBuffer(dev, (n, K + 1, nX)), lib.DeviceBuffer(dev, (n, K, nU))
                    b["st"], b["cost"] = lib.DeviceBuffer(dev, (n,), np.int32), lib.DeviceBuffer(dev, (n,))
                    params = None
                    if par is not None:
                        V = par[1] if par[1].shape[0] == 1 else par[1][np.repeat(rows[g], M)]
                        b["params"] = up(np.ascontiguousarray(np.broadcast_to(V, (n, V.shape[1]))))
                        params = (par[0], b["params"])
                    sys_.project_raw(True, n, K, float(ds.time[0]), float(ds.time[1] - ds.time[0]), b["bX"], b["bU"],
                                     b["Kc"], b["pX"], b["pU"], b["st"], k_per_instance=True, use_hint=False,
                                     tolerance=ds.varint.tolerance, times=times, params=params)
                    ref = self._ref_rows(np.repeat(rows[g], M))
                    b["ref"] = None if ref is None else up(ref, np.int32)
                    lib.track_raw(True, dev, n, K, nX, nU, nref=d["nref"], X=b["pX"], U=b["pU"], Xd=d["Xd"], Ud=d["Ud"],
                                  Q=d["Qc"], R=d["Rc"], ref_index=b["ref"], cost=b["cost"])
                    st, c1 = b["st"].download(), b["cost"].download()
                    left = []
                    for gi, r in enumerate(g):
                        for i, m in enumerate(ms):
                            j = gi * M + i
                            if st[j] != 0:
                                continue      # a failed simulation is skipped, as armijo_simulate's exception is
                            if c1[j] < cost0[r] + self.armijo_alpha * lam[i] * dcost0[r]:
                                Xn[r], Un[r] = b["pX"].download_row(j), b["pU"].download_row(j)
                                cost[r], macc[r] = c1[j], m
                                break
                        else:
                            left.append(r)
                    g = np.asarray(left, dtype=np.int64)
                    m0 += M
                finally:
                    ds._free(b)
            status[g] = ARMIJO_FAILED
        finally:
            times.free()
        return Xn, Un, cost, status, macc

    def armijo_search(self, X, U, Kproj, dX, dU):
        """DOptimizer.armijo_search on the GPU.  One trajectory: (nX, nU, cost), ConvergenceError when no step size
        passes.  R rollouts: (nX, nU, cost [R]); a rollout whose search fails keeps its trajectory and cost0, and
        last_status marks it ARMIJO_FAILED (last_armijo_m holds the accepted m, -1 for none)."""
        from . import lib
        single, Xb, Ub = self._batch(X, U)
        _, dXb, dUb = self._batch(dX, dU)
        Rn, K = Xb.shape[0], Xb.shape[1] - 1
        Kp = np.asarray(Kproj, float)
        Kp = np.ascontiguousarray(np.broadcast_to(Kp, (Rn,) + Kp.shape[-3:]))
        dev = self.dsys.varint.sys.device
        rows = np.arange(Rn)
        d = {}
        try:
            self._upload_cost(d, Xb, Ub, self._ref_rows(rows))
            up = lambda a: lib.DeviceBuffer(dev, a.shape).upload(np.ascontiguousarray(a))
            d["dX"], d["dU"], d["K"] = up(-dXb), up(-dUb), up(Kp)
            d["cost"] = lib.DeviceBuffer(dev, (Rn,))
            lib.track_raw(True, dev, Rn, K, self.dsys.nX, self.dsys.nU, nref=d["nref"], X=d["X"], U=d["U"], Xd=d["Xd"],
                          Ud=d["Ud"], Q=d["Qc"], R=d["Rc"], ref_index=d["ref_index"], cost=d["cost"])
            dcost0 = self._dcost_on_device(d, Rn, K)
            cost0 = d["cost"].download()
            Xn, Un, cost, status, macc = self._search(d, Xb, Ub, rows, rows, cost0, dcost0)
        finally:
            self.dsys._free(d)
        self.last_status, self.last_armijo_m = status, macc
        if single:
            if status[0] != 0:
                raise ConvergenceError("Armijo Failed to Converge", status)
            return self.armijo_search_return(Xn[0], Un[0], float(cost[0]))
        return self.armijo_search_return(Xn, Un, cost)

    def _step(self, Xb, Ub, rows, method):
        """One step of rollouts `rows` (their trajectories Xb / Ub): (converged, X, U, dcost0, cost, status, m)."""
        Rn, K = Xb.shape[0], Xb.shape[1] - 1
        d = self._direction(Xb, Ub, rows, method)
        try:
            dcost0 = self._dcost_on_device(d, Rn, K)
            cost0 = d["cost"].download()
            conv = np.abs(dcost0) < self.descent_tolerance
            Xn, Un, cost, status, macc = self._search(d, Xb, Ub, rows, np.flatnonzero(~conv), cost0, dcost0)
        finally:
            self.dsys._free(d)
        status[conv] = STEP_CONVERGED
        return conv, Xn, Un, dcost0, cost, status, macc

    def step(self, iteration, X, U, method="steepest"):
        """DOptimizer.step: the descent direction, cost0 and dcost0, then (unless |dcost0| < descent_tolerance) the
        Armijo search.  Returns (converged, X, U, dcost0, cost); with R rollouts each is per rollout, and last_status
        holds STEP_ACCEPTED, STEP_CONVERGED or ARMIJO_FAILED (the trajectory kept).  One trajectory raises
        ConvergenceError when its search fails."""
        single, Xb, Ub = self._batch(X, U)
        conv, Xn, Un, dcost0, cost, status, macc = self._step(Xb, Ub, np.arange(Xb.shape[0]), method)
        self.last_status, self.last_armijo_m = status, macc
        if single:
            if status[0] == ARMIJO_FAILED:
                raise ConvergenceError("Armijo Failed to Converge", status)
            return self.step_return(bool(conv[0]), Xn[0], Un[0], float(dcost0[0]), float(cost[0]))
        return self.step_return(conv, Xn, Un, dcost0, cost)

    def optimize(self, X, U, max_steps=50):
        """DOptimizer.optimize: project (X, U) onto a trajectory of the system, then steps with first_method for
        first_method_iterations steps and second_method afterwards.  Each rollout is frozen once it converges or its
        Armijo search fails; last_status holds STEP_CONVERGED, ARMIJO_FAILED or STEP_ACCEPTED (max_steps reached).
        Returns (converged, X, U); one trajectory raises ConvergenceError when its search fails."""
        if self.optimize_ic:
            raise ValueError("optimize_ic=True is not supported")
        single, Xb, Ub = self._batch(X, U)
        Xb, Ub = self.dsys.project(Xb, Ub, self.dsys.calc_feedback_controller(Xb, Ub))
        Xb, Ub = Xb.copy(), Ub.copy()
        status = np.zeros(Xb.shape[0], np.int32)
        live = np.arange(Xb.shape[0])
        method = self.first_method
        for i in range(max_steps):
            if i == self.first_method_iterations:
                method = self.second_method
            if not live.size:
                break
            _, Xn, Un, _, _, st, _ = self._step(Xb[live], Ub[live], live, method)
            Xb[live], Ub[live] = Xn, Un
            status[live] = st
            live = live[st == STEP_ACCEPTED]
        self.last_status = status
        converged = status == STEP_CONVERGED
        if single:
            if status[0] == ARMIJO_FAILED:
                raise ConvergenceError("Armijo Failed to Converge", status)
            return bool(converged[0]), Xb[0], Ub[0]
        return converged, Xb, Ub
