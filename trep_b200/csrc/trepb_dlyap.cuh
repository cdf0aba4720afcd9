// Closed-loop cost and stability of stationary gains: the discrete Lyapunov (Stein) equation, batched over
// (gain, model) pairs,
//
//     P = A_c^T P A_c + Q_c,     A_c = A - B K,     Q_c = Q - S K - K^T S^T + K^T R K
//
// (u = -K x under the stage cost x^T Q x + 2 x^T S u + u^T R u), by Smith's doubling: from P = Q_c, F = A_c,
//
//     P <- P + F^T P F,   F <- F F
//
// so that after k steps P = sum_{i < 2^k} (A_c^T)^i Q_c A_c^i and F = A_c^(2^k).  Stop when ||P' - P||_F <= tol ||P'||_F
// and ||F'||_F <= tol.  The test on F is the stability certificate: F -> 0 exactly when rho(A_c) < 1, and then
// P_inf - P' = F'^T P_inf F', so the second test alone bounds P's relative error by tol^2.  Without it a Q_c that is
// zero on an unstable direction would "converge" to a P that means nothing.  P is then accepted only if
// ||A_c^T P A_c - P + Q_c||_F <= 1e-6 ||[A_c^T P A_c, P, Q_c]||_F, the DARE's acceptance test (trepb_dare.cuh).
//
// One CTA per pair (grid-stride over the batch, as dare_kernel); pair r evaluates gain gidx[r] under model midx[r]
// (either index may be null: gain r / model r).  Shared memory:
//   Ac  [n][ld]   A_c, kept for the residual
//   P   [n][ld]   the iterate P, full (the upper triangle is computed and mirrored)
//   F   [n][ld]   the iterate F, at the end Q_c again
//   T   [wk]      R K [nU][n] in the set-up; P F, then F F, after which F and T swap pointers (so during the
//                 doubling either block plays either role, and only n ld doubles of T are used); at the end, back
//                 at this block, R K, then P A_c  (wk = max(n ld, nU n))
// (ld = (n + 1) | 1: odd, so walks down a column are free of bank conflicts), and the per-warp partial norms.  No
// product overwrites an operand, so every element is one thread's dot product.  4 n ld + 3 nw doubles or so: 208 KB at
// nX = 80, and no more than dare_kernel asks for at any shape.
//
// Every output element is summed by one thread in ascending index order, the norms are reduced in an order fixed by the
// shape, and Q_c / A_c are formed the same way in the set-up and for the residual, so a pair gives the same bits alone
// and inside any batch.  P is mirrored from its upper triangle, so it is symmetric bit for bit.
#pragma once
#include <cuda_runtime.h>

namespace trepb {
namespace {

struct DlyapParams {
    long long pairs, G, M;             // pairs, gains in K, models in A / B
    int nX, nU, max_it;
    double tol;
    const double *A, *B, *K, *Q, *R, *S;   // [M][nX][nX], [M][nX][nU], [G][nU][nX]; Q / R / S at stride Qs / Rs / Ss
    long long Qs, Rs, Ss;                  // (per model; 0: shared)
    const int *gidx, *midx;            // [pairs] or null
    const double *x0, *W;              // x0 [nX] at stride xs per pair, W [nX][nX]; both null: no cost
    long long xs;
    double *P, *cost;                  // [pairs][nX][nX], [pairs], either may be null
    int *status, *iters;               // [pairs], iters may be null
};

// Shared-memory layout in doubles, for the launcher and the kernel alike.
struct DlyapLayout {
    int ld, nw;                         // leading dimension of the n x n blocks, warps per CTA
    long long Ac, P, F, T, red, total;
};
__host__ __device__ __forceinline__ DlyapLayout dlyap_layout(int n, int m) {
    DlyapLayout L;
    L.ld = (n + 1) | 1;
    const long long nw = ((long long)n * n + 255) / 256;
    L.nw = (int)(nw < 2 ? 2 : nw > 16 ? 16 : nw);
    const long long blk = (long long)n * L.ld, rk = (long long)m * n;
    L.Ac = 0;
    L.P = blk;
    L.F = 2 * blk;
    L.T = 3 * blk;
    L.red = L.T + (blk > rk ? blk : rk);
    L.total = L.red + 3LL * L.nw;
    return L;
}

// Block-wide reduction of three per-thread partial sums in an order fixed by the shape: warp shuffles, then every
// thread adds the warps' sums in ascending order after the barrier (so each gets the same bits, and no second barrier
// is needed: red is written again only after further barriers).
__device__ __forceinline__ void dlyap_reduce3(double& a, double& b, double& c, double* red, int nw) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
        c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    if (lane == 0) { red[warp] = a; red[nw + warp] = b; red[2 * nw + warp] = c; }
    __syncthreads();
    a = b = c = 0.0;
    for (int w = 0; w < nw; ++w) { a += red[w]; b += red[nw + w]; c += red[2 * nw + w]; }
}

// Q_c = (Q + Q^T)/2 - S K - K^T S^T + K^T (R + R^T)/2 K into Qc [n][ld] (upper triangle computed, mirrored), through
// RK = (R + R^T)/2 K [m][n] in T.  Ends with a barrier.
__device__ void dlyap_qc(double* Qc, int ld, double* T, const double* Q, const double* R, const double* S,
                         const double* K, int n, int m) {
    const int tid = threadIdx.x, nth = blockDim.x;
    for (int e = tid; e < m * n; e += nth) {
        const int c = e / n, j = e - c * n;
        double acc = 0.0;
        for (int d = 0; d < m; ++d) acc += (0.5 * (R[c * m + d] + R[d * m + c])) * K[d * n + j];
        T[e] = acc;
    }
    __syncthreads();
    for (int e = tid; e < n * n; e += nth) {
        const int i = e / n, j = e - i * n;
        if (j < i) continue;
        double acc = 0.5 * (Q[e] + Q[j * n + i]);
        if (S) {
            double sk = 0.0;
            for (int c = 0; c < m; ++c) sk += S[i * m + c] * K[c * n + j] + K[c * n + i] * S[j * m + c];
            acc -= sk;
        }
        double kr = 0.0;
        for (int c = 0; c < m; ++c) kr += K[c * n + i] * T[c * n + j];
        acc += kr;
        Qc[i * ld + j] = acc;
        Qc[j * ld + i] = acc;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(512, 1) dlyap_kernel(const DlyapParams p) {
    extern __shared__ __align__(16) double lsm[];
    const int n = p.nX, m = p.nU, tid = threadIdx.x, nth = blockDim.x;
    const DlyapLayout L = dlyap_layout(n, m);
    const int ld = L.ld, nw = L.nw;
    double* Ac = lsm + L.Ac;
    double* Pb = lsm + L.P;
    double* red = lsm + L.red;
    const double big = 1.7976931348623157e308, tol2 = p.tol * p.tol;
    for (long long r = blockIdx.x; r < p.pairs; r += gridDim.x) {
        const long long gi = p.gidx ? (long long)p.gidx[r] : r, mi = p.midx ? (long long)p.midx[r] : r;
        double* F = lsm + L.F;
        double* T = lsm + L.T;
        int state = 0, it = 0;              // 0 iterating, 1 converged, else the failure status
        if (gi < 0 || gi >= p.G || mi < 0 || mi >= p.M) state = TREPB_DLYAP_BAD_INDEX;
        const double* Am = p.A + mi * n * n;
        const double* Bm = p.B + mi * n * m;
        const double* Kg = p.K + gi * m * n;
        const double* Qm = p.Q + mi * p.Qs;
        const double* Rm = p.R + mi * p.Rs;
        const double* Sm = p.S ? p.S + mi * p.Ss : nullptr;
        if (state == 0) {
            // ---- set-up: P = Q_c, A_c = F = A - B K ----------------------------------------------------------------
            for (int e = tid; e < n * n; e += nth) {
                const int i = e / n, j = e - i * n;
                double bk = 0.0;
                for (int c = 0; c < m; ++c) bk += Bm[i * m + c] * Kg[c * n + j];
                const double a = Am[e] - bk;
                Ac[i * ld + j] = a;
                F[i * ld + j] = a;
            }
            dlyap_qc(Pb, ld, T, Qm, Rm, Sm, Kg, n, m);
        }
        // ---- doubling ------------------------------------------------------------------------------------------------
        while (state == 0) {
            ++it;
            // T = P F
            for (int e = tid; e < n * n; e += nth) {
                const int i = e / n, j = e - i * n;
                double acc = 0.0;
                for (int k = 0; k < n; ++k) acc += Pb[i * ld + k] * F[k * ld + j];
                T[i * ld + j] = acc;
            }
            __syncthreads();
            // P += F^T T (upper triangle, mirrored; the change of P and P itself summed up)
            double d2 = 0.0, p2 = 0.0, f2 = 0.0;
            for (int e = tid; e < n * n; e += nth) {
                const int i = e / n, j = e - i * n;
                if (j < i) continue;
                double acc = 0.0;
                for (int k = 0; k < n; ++k) acc += F[k * ld + i] * T[k * ld + j];
                const double p0 = Pb[i * ld + j], p1 = p0 + acc, dp = p1 - p0, w = j == i ? 1.0 : 2.0;
                Pb[i * ld + j] = p1;
                Pb[j * ld + i] = p1;
                d2 += w * (dp * dp);
                p2 += w * (p1 * p1);
            }
            __syncthreads();
            // T = F F, then T is the new F
            for (int e = tid; e < n * n; e += nth) {
                const int i = e / n, j = e - i * n;
                double acc = 0.0;
                for (int k = 0; k < n; ++k) acc += F[i * ld + k] * F[k * ld + j];
                T[i * ld + j] = acc;
                f2 += acc * acc;
            }
            double* const t = F;
            F = T;
            T = t;
            dlyap_reduce3(d2, p2, f2, red, nw);
            if (!(d2 <= big && p2 <= big && f2 <= big)) state = TREPB_DLYAP_NONFINITE;
            else if (d2 <= tol2 * p2 && f2 <= tol2) state = 1;
            else if (it >= p.max_it) state = TREPB_DLYAP_NOT_CONVERGED;
        }
        // ---- acceptance: ||A_c^T P A_c - P + Q_c||_F <= 1e-6 ||[A_c^T P A_c, P, Q_c]||_F ----------------------------
        if (state == 1) {
            // back to the fixed blocks: after an odd number of squarings T is F's n ld block, too small for R K
            // when nU n > n ld; the last F is no longer needed
            F = lsm + L.F;
            T = lsm + L.T;
            dlyap_qc(F, ld, T, Qm, Rm, Sm, Kg, n, m);
            for (int e = tid; e < n * n; e += nth) {   // T = P A_c
                const int i = e / n, j = e - i * n;
                double acc = 0.0;
                for (int k = 0; k < n; ++k) acc += Pb[i * ld + k] * Ac[k * ld + j];
                T[i * ld + j] = acc;
            }
            __syncthreads();
            double r2 = 0.0, t2 = 0.0, unused = 0.0;
            for (int e = tid; e < n * n; e += nth) {
                const int i = e / n, j = e - i * n;
                double apa = 0.0;
                for (int k = 0; k < n; ++k) apa += Ac[k * ld + i] * T[k * ld + j];
                const double pij = Pb[i * ld + j], qij = F[i * ld + j], v = apa - pij + qij;
                r2 += v * v;
                t2 += apa * apa + pij * pij + qij * qij;
            }
            dlyap_reduce3(r2, t2, unused, red, nw);
            if (!(r2 <= big && t2 <= big)) state = TREPB_DLYAP_NONFINITE;
            else if (!(r2 <= 1e-12 * t2)) state = TREPB_DLYAP_NOT_CONVERGED;
        }
        // ---- outputs: P, cost = x0^T P x0 or trace(P W) (one thread per row, then one thread over the rows) --------
        double* v = T;                       // free once the residual is reduced
        if (state == 1) {
            if (p.P)
                for (int e = tid; e < n * n; e += nth) p.P[r * n * n + e] = Pb[(e / n) * ld + e % n];
            if (p.cost) {
                const double* x = p.x0 ? p.x0 + r * p.xs : nullptr;
                for (int i = tid; i < n; i += nth) {
                    double acc = 0.0;
                    if (x)
                        for (int j = 0; j < n; ++j) acc += Pb[i * ld + j] * x[j];
                    else
                        for (int j = 0; j < n; ++j) acc += Pb[i * ld + j] * p.W[j * n + i];
                    v[i] = acc;
                }
                __syncthreads();
            }
        }
        if (tid == 0) {
            if (p.cost) {
                double c = __longlong_as_double(0x7ff0000000000000LL);   // +inf: no finite cost is certified
                if (state == 1) {
                    const double* x = p.x0 ? p.x0 + r * p.xs : nullptr;
                    c = 0.0;
                    for (int i = 0; i < n; ++i) c += x ? x[i] * v[i] : v[i];
                }
                p.cost[r] = c;
            }
            p.status[r] = state == 1 ? TREPB_DLYAP_STABLE : state;
            if (p.iters) p.iters[r] = it;
        }
        __syncthreads();
    }
}

}  // namespace
}  // namespace trepb
