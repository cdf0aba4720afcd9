"""TEST INFRASTRUCTURE: host references of the device's Riccati / LQ solve (trepb_lqr.cu) and of its tangent and
adjoint sweeps (trepb_sweep.cuh), written out from the recurrences in those files' header comments.  Never imported
by the product.

- `solve_tv_lq_ld`, `tangent_ld`, `adjoint_ld`: one rollout in np.longdouble (x87 80-bit extended precision on
  x86-64), the yardstick for the fp64 kernels.  numpy's long-double matmul does not use BLAS, so a step costs
  O(nX^3) in plain loops: use these on a sample of rollouts and on short horizons.
- `solve_tv_lq_f64`: the same recurrence in fp64 over a whole batch at once (numpy's batched solve), to check
  thousands of rollouts quickly."""
import numpy as np

LD = np.longdouble


def _ld(x):
    return None if x is None else np.array(x, dtype=LD)


def solve_ld(G, M):
    """G^-1 M in long double by Gaussian elimination with partial pivoting, every column of M a right-hand side.
    np.linalg.solve does not take long double.  Raises np.linalg.LinAlgError on an exactly zero pivot."""
    n = G.shape[0]
    a = np.concatenate([np.array(G, dtype=LD), np.array(M, dtype=LD)], axis=1)
    for k in range(n):
        p = k + int(np.argmax(np.abs(a[k:, k])))
        if a[p, k] == 0:
            raise np.linalg.LinAlgError("singular gamma")
        if p != k:
            a[[k, p]] = a[[p, k]]
        a[k + 1:] -= np.outer(a[k + 1:, k] / a[k, k], a[k])
    x = a[:, n:]
    for k in reversed(range(n)):
        x[k] = (x[k] - a[k, k + 1:n] @ x[k + 1:]) / a[k, k]
    return x


def solve_tv_lq_ld(A, B, Q, R, S=None, q=None, r=None, gammas=None):
    """One rollout of trepb_lq_batch (q, r given) or trepb_lqr_batch (q = r = None):

        P = Q(K), b = q[K];  for k = K-1 .. 0:
            gamma = R(k) + B^T P B;  Kp = B^T P A (+ S[k]^T);  g = r[k] + B^T b (0 without q, r)
            [K[k] | C[k]] = gamma^-1 [Kp | g]
            P = Q(k) + A^T P A - Kp^T K[k];  P = (P + P^T) / 2;  b = q[k] + A^T b - K[k]^T g

    A [K,nX,nX], B [K,nX,nU]; Q [nX,nX] (shared by every step) or [K+1,nX,nX]; R [nU,nU] or [K,nU,nU]; S [K,nX,nU]
    or None; q [K+1,nX], r [K,nU].  Returns (K [K,nU,nX], C [K,nU] or None, P0 [nX,nX], b0 [nX] or None) in long
    double.  `gammas`, a list, receives every step's gamma (k descending)."""
    A, B, Q, R, S, q, r = (_ld(x) for x in (A, B, Q, R, S, q, r))
    n, nX, nU = A.shape[0], A.shape[1], B.shape[2]
    Qk = (lambda k: Q[k]) if Q.ndim == 3 else (lambda k: Q)
    Rk = (lambda k: R[k]) if R.ndim == 3 else (lambda k: R)
    affine = q is not None
    Kf = np.zeros((n, nU, nX), LD)
    Cf = np.zeros((n, nU), LD) if affine else None
    P = Qk(n).copy()
    b = q[n].copy() if affine else None
    for k in reversed(range(n)):
        a, bk = A[k], B[k]
        gamma = Rk(k) + bk.T @ P @ bk
        Kp = bk.T @ P @ a
        if S is not None:
            Kp = Kp + S[k].T
        g = r[k] + bk.T @ b if affine else np.zeros(nU, LD)
        if gammas is not None:
            gammas.append(gamma)
        X = solve_ld(gamma, np.concatenate([Kp, g[:, None]], axis=1))
        Kf[k] = X[:, :nX]
        P = Qk(k) + a.T @ P @ a - Kp.T @ Kf[k]
        P = (P + P.T) / 2
        if affine:
            Cf[k] = X[:, nX]
            b = q[k] + a.T @ b - Kf[k].T @ g
    return Kf, Cf, P, b


def solve_tv_lq_f64(A, B, Q, R, S=None, q=None, r=None):
    """The recurrence of solve_tv_lq_ld in fp64 over a batch: A [N,K,nX,nX], B [N,K,nX,nU]; every cost array with a
    per-step axis and a leading axis of N or 1 (Q [N|1,K+1,nX,nX], R [N|1,K,nU,nU], S [N|1,K,nX,nU] or None,
    q [N|1,K+1,nX], r [N|1,K,nU], q = r = None for the LQR).  Returns (K, C or None, P0, b0 or None)."""
    N, n, nX, nU = A.shape[0], A.shape[1], A.shape[2], B.shape[3]
    affine = q is not None
    Kf = np.zeros((N, n, nU, nX))
    Cf = np.zeros((N, n, nU)) if affine else None
    P = np.broadcast_to(Q[:, n], (N, nX, nX)).copy()
    b = np.broadcast_to(q[:, n], (N, nX)).copy() if affine else None
    for k in reversed(range(n)):
        a, bk = A[:, k], B[:, k]
        bt = np.swapaxes(bk, 1, 2)
        gamma = R[:, k] + bt @ P @ bk
        Kp = bt @ P @ a
        if S is not None:
            Kp = Kp + np.swapaxes(S[:, k], 1, 2)
        g = (r[:, k] + np.einsum("nxu,nx->nu", bk, b)) if affine else np.zeros((N, nU))
        X = np.linalg.solve(gamma, np.concatenate([Kp, g[:, :, None]], axis=2))
        Kf[:, k] = X[:, :, :nX]
        P = Q[:, k] + np.swapaxes(a, 1, 2) @ P @ a - np.swapaxes(Kp, 1, 2) @ Kf[:, k]
        P = (P + np.swapaxes(P, 1, 2)) / 2
        if affine:
            Cf[:, k] = X[:, :, nX]
            b = q[:, k] + np.einsum("nxy,nx->ny", a, b) - np.einsum("nux,nu->nx", Kf[:, k], g)
    return Kf, Cf, P, b


def tangent_ld(A, B=None, K=None, bdX=None, bdU=None, x0=None):
    """One rollout of trepb_tangent_batch:
        dX[0] = x0 (default bdX[0], or zero);  dU[k] = bdU[k] - K[k] (dX[k] - bdX[k]);  dX[k+1] = A[k] dX[k] + B[k] dU[k]
    A [K,nX,nX], B [K,nX,nU] and K [K,nU,nX] (None: no inputs), bdX [K+1,nX], bdU [K,nU], x0 [nX]; a None vector is
    zero.  Returns (dX [K+1,nX], dU [K,nU]) in long double."""
    A, B, K, bdX, bdU, x0 = (_ld(x) for x in (A, B, K, bdX, bdU, x0))
    n, nX = A.shape[0], A.shape[1]
    nU = 0 if B is None else B.shape[2]
    dX, dU = np.zeros((n + 1, nX), LD), np.zeros((n, nU), LD)
    dX[0] = x0 if x0 is not None else bdX[0] if bdX is not None else 0
    for k in range(n):
        if nU:
            e = dX[k] - bdX[k] if bdX is not None else dX[k]
            dU[k] = (bdU[k] if bdU is not None else 0) - K[k] @ e
            dX[k + 1] = A[k] @ dX[k] + B[k] @ dU[k]
        else:
            dX[k + 1] = A[k] @ dX[k]
    return dX, dU


def adjoint_ld(A, m_dx, B=None, K=None, l_dx=None, l_du=None):
    """One rollout of trepb_adjoint_batch:
        z[K] = m_dx;  z[k] = l_dx[k] + A[k]^T z[k+1] - K[k]^T (l_du[k] + B[k]^T z[k+1])
    (K None: the open-loop costate z[k] = l_dx[k] + A[k]^T z[k+1]; l_du is then unused).  A [K,nX,nX], m_dx [nX],
    B [K,nX,nU], K [K,nU,nX], l_dx [K,nX], l_du [K,nU]; a None vector is zero.  Returns z [K+1,nX] in long double;
    the kernel's optional z1 output is z[1:]."""
    A, m_dx, B, K, l_dx, l_du = (_ld(x) for x in (A, m_dx, B, K, l_dx, l_du))
    n, nX = A.shape[0], A.shape[1]
    z = np.zeros((n + 1, nX), LD)
    z[n] = m_dx
    for k in reversed(range(n)):
        v = A[k].T @ z[k + 1]
        if l_dx is not None:
            v = l_dx[k] + v
        if K is not None and K.shape[1] > 0:
            g = B[k].T @ z[k + 1]
            if l_du is not None:
                g = l_du[k] + g
            v = v - K[k].T @ g
        z[k] = v
    return z
