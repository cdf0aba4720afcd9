// Stationary discrete LQR: the stabilizing solution of the discrete algebraic Riccati equation, batched over models,
//
//     P = A^T P A - (A^T P B + S)(R + B^T P B)^-1 (B^T P A + S^T) + Q,     K = (R + B^T P B)^-1 (B^T P A + S^T)
//
// (u = -K x), by the structure-preserving doubling algorithm (SDA; Chu, Fan, Lin and Wang 2004).  The cross term is
// folded in first (A <- A - B R^-1 S^T, Q <- Q - S R^-1 S^T), then from G = B R^-1 B^T, H = Q
//
//     W = I + G H,   A' = A W^-1 A,   G' = G + A W^-1 G A^T,   H' = H + A^T H W^-1 A
//
// until ||H' - H||_F <= tol ||H'||_F: H converges quadratically to P, and A need not be invertible.  K is then formed
// from P and the caller's A, B, R, S, and P is accepted only if it satisfies the equation (relative residual <= 1e-6:
// without a stabilizing solution the doubling can stall on a matrix that does not, see below).
//
// One CTA per model (grid-stride over the batch, as lqr_kernel), every matrix in shared memory:
//   A   [n][ld]   the doubling iterate A_k
//   GH  [n][ld]   G_k and H_k, both symmetric, packed: G(i, j) at [i][j] for j <= i, H(i, j) at [i][j + 1] for j >= i
//   W1  [n][ld]   W, then the packed pair Z = W^-1 G (lower) / Y = H W^-1 (upper), both symmetric
//   W2  [n][ld]   W^-1, then X = W^-1 A
// (ld = (n + 1) | 1: odd, so walks down a column are free of bank conflicts), one row buffer of n doubles per warp,
// and the pivot buffers of the eliminations.  W1 / W2 also hold the set-up (B, S, R and [B^T | S^T]) and the gain
// solve ([R + B^T P B | B^T P A + S^T]).  The products whose result overwrites an operand (X = W^-1 A over W^-1,
// A' = A X over A, G' and H' over GH) run row by row, one warp per row staging the row it reads in its buffer; all
// others write a block no one reads.  4 n ld + 18 n doubles or so: 216 KB for the marionette's nX = 80.
//
// Every output element is summed by one thread in ascending index order, the eliminations use a fixed pivot rule,
// and the stopping test's norms are reduced in an order fixed by the shape, so a model gives the same bits alone and
// inside any batch.  P is mirrored from one triangle, so it is symmetric bit for bit.
#pragma once
#include <cuda_runtime.h>

namespace trepb {
namespace {

struct DareParams {
    long long batch;
    int nX, nU, max_it;
    double tol;
    const double *A, *B, *Q, *R, *S;   // [batch][nX][nX], [batch][nX][nU], Q / R / S at stride Qs / Rs / Ss (0: shared)
    long long Qs, Rs, Ss;
    double *K, *P;                     // [batch][nU][nX], [batch][nX][nX], either may be null
    int *status, *iters;               // [batch], iters may be null
};

// Shared-memory layout in doubles, for the launcher and the kernel alike.
struct DareLayout {
    int ld, nw;                         // leading dimension of the n x n blocks, warps per CTA
    long long A, GH, W1, W2, rows, g, prow, krow, red, total;
};
__host__ __device__ __forceinline__ DareLayout dare_layout(int n, int m) {
    DareLayout L;
    L.ld = (n + 1) | 1;
    const long long s = n > m ? n : m;
    long long nw = (s * s + 255) / 256;
    L.nw = (int)(nw < 2 ? 2 : nw > 16 ? 16 : nw);
    const long long blk = (long long)n * L.ld;
    // W1 + W2 also hold the set-up: B, S [n][m], R [m][m], [B^T | S^T] [m][2n]  (the gain solve needs less)
    long long wk = 2 * blk;
    const long long setup = 4LL * n * m + (long long)m * m;
    if (setup > wk) wk = setup;
    L.A = 0;
    L.GH = blk;
    L.W1 = 2 * blk;
    L.W2 = 3 * blk;                     // = W1 + blk; the set-up runs over W1 .. W1 + wk
    L.rows = 2 * blk + wk;
    L.g = L.rows + (long long)L.nw * n;
    L.prow = L.g + s;
    L.krow = L.prow + 2LL * n + m;      // widest elimination: [R | B^T | S^T], m + 2n columns
    L.red = L.krow + 2LL * n + m;
    L.total = L.red + 2LL * L.nw + 2;
    return L;
}

// L [n][ldl] is reduced to the identity by Gauss-Jordan elimination with partial pivoting (largest |L[r][k]| among
// the rows r >= k, the lowest row among equals; rows are exchanged), and every row operation is applied to Rt
// [n][ldr] (nr columns): Rt <- L^-1 Rt.  Every warp finds the pivot on its own; the pivot row, the row it replaces
// and the multipliers are staged in g / prow / krow, so each element then takes one update with no race.  Columns
// <= k of L are left as they are (never read again).  Returns false (on every thread) for an exact zero pivot.
__device__ bool dare_gj(double* L, int ldl, double* Rt, int ldr, int n, int nr, double* g, double* prow, double* krow) {
    const int tid = threadIdx.x, nth = blockDim.x, lane = tid & 31;
    for (int k = 0; k < n; ++k) {
        double best = 0.0;
        int br = 0x7fffffff;
        for (int r = k + lane; r < n; r += 32) {
            const double v = fabs(L[r * ldl + k]);
            if (v > best) { best = v; br = r; }
        }
        const unsigned long long bits = (unsigned long long)__double_as_longlong(best);
        const unsigned hi = (unsigned)(bits >> 32), lo = (unsigned)bits;
        const unsigned mh = __reduce_max_sync(0xffffffffu, hi);
        const unsigned ml = __reduce_max_sync(0xffffffffu, hi == mh ? lo : 0u);
        const int p = (int)__reduce_min_sync(0xffffffffu, (hi == mh && lo == ml) ? (unsigned)br : 0x7fffffffu);
        if (mh == 0u && ml == 0u) return false;
        const double rinv = 1.0 / L[p * ldl + k];
        const int nl = n - k - 1, nc = nl + nr;
        for (int e = tid; e < nc; e += nth) {
            prow[e] = e < nl ? L[p * ldl + k + 1 + e] : Rt[p * ldr + e - nl];
            krow[e] = e < nl ? L[k * ldl + k + 1 + e] : Rt[k * ldr + e - nl];
        }
        for (int i = tid; i < n; i += nth) {
            const int si = i == k ? p : i == p ? k : i;
            g[i] = L[si * ldl + k] * rinv;
        }
        __syncthreads();
        // row k <- prow / pivot; row p <- krow - g[p] prow; any other row i <- row i - g[i] prow
        for (int e = tid; e < n * nc; e += nth) {
            const int i = e / nc, c = e - i * nc;
            double* d = c < nl ? L + i * ldl + k + 1 + c : Rt + i * ldr + c - nl;
            if (i == k) *d = prow[c] * rinv;
            else *d = (i == p ? krow[c] : *d) - g[i] * prow[c];
        }
        __syncthreads();
    }
    return true;
}

// G(i, j) and H(i, j) of the packed pair (also Z and Y of W1)
__device__ __forceinline__ double dare_lo(const double* M, int ld, int i, int j) { return i >= j ? M[i * ld + j] : M[j * ld + i]; }
__device__ __forceinline__ double dare_up(const double* M, int ld, int i, int j) { return i <= j ? M[i * ld + j + 1] : M[j * ld + i + 1]; }

__global__ void __launch_bounds__(512, 1) dare_kernel(const DareParams p) {
    extern __shared__ __align__(16) double dsm[];
    const int n = p.nX, m = p.nU, tid = threadIdx.x, nth = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const DareLayout L = dare_layout(n, m);
    const int ld = L.ld, nw = L.nw;
    double* Ab = dsm + L.A;
    double* GH = dsm + L.GH;
    double* W1 = dsm + L.W1;
    double* W2 = dsm + L.W2;
    double* rb = dsm + L.rows + (long long)warp * n;   // this warp's row buffer
    double* g = dsm + L.g;
    double* prow = dsm + L.prow;
    double* krow = dsm + L.krow;
    double* red = dsm + L.red;
    __shared__ int s_state;                             // 0 iterating, 1 converged, else the failure status
    for (long long r = blockIdx.x; r < p.batch; r += gridDim.x) {
        const double* Ar = p.A + r * n * n;
        const double* Br = p.B + r * n * m;
        const double* Qr = p.Q + r * p.Qs;
        const double* Rr = p.R + r * p.Rs;
        const double* Sr = p.S ? p.S + r * p.Ss : nullptr;
        // ---- set-up: [B^T | S^T] <- R^-1 [B^T | S^T], G = B R^-1 B^T, A -= B R^-1 S^T, H = Q - S R^-1 S^T ----
        double* Bs = W1;                     // [n][m]
        double* Ss = Bs + n * m;             // [n][m]
        double* Rg = Ss + n * m;             // [m][m]
        double* Rt = Rg + m * m;             // [m][2n]
        const int ncol = Sr ? 2 * n : n;
        for (int e = tid; e < n * n; e += nth) {
            const int i = e / n, j = e - i * n;
            Ab[i * ld + j] = Ar[e];
            if (j >= i) GH[i * ld + j + 1] = 0.5 * (Qr[e] + Qr[j * n + i]);
        }
        for (int e = tid; e < n * m; e += nth) {
            const int i = e / m, c = e - i * m;
            Bs[e] = Br[e];
            Rt[c * 2 * n + i] = Br[e];
            if (Sr) { Ss[e] = Sr[e]; Rt[c * 2 * n + n + i] = Sr[e]; }
        }
        for (int e = tid; e < m * m; e += nth) Rg[e] = Rr[e];
        if (tid == 0) s_state = 0;
        __syncthreads();
        int it = 0;
        if (!dare_gj(Rg, m, Rt, 2 * n, m, ncol, g, prow, krow)) {
            if (tid == 0) s_state = TREPB_DARE_SINGULAR;
        } else {
            for (int e = tid; e < n * n; e += nth) {
                const int i = e / n, j = e - i * n;
                if (j <= i) {
                    double acc = 0.0;
                    for (int c = 0; c < m; ++c) acc += Bs[i * m + c] * Rt[c * 2 * n + j];
                    GH[i * ld + j] = acc;
                }
                if (Sr) {
                    double acc = 0.0;
                    for (int c = 0; c < m; ++c) acc += Bs[i * m + c] * Rt[c * 2 * n + n + j];
                    Ab[i * ld + j] -= acc;
                    if (j >= i) {
                        double h = 0.0;
                        for (int c = 0; c < m; ++c) h += Ss[i * m + c] * Rt[c * 2 * n + n + j];
                        GH[i * ld + j + 1] -= h;
                    }
                }
            }
        }
        __syncthreads();
        // ---- doubling ----------------------------------------------------------------------------------------------
        while (s_state == 0) {
            ++it;
            // W1 = I + G H, W2 = I
            for (int e = tid; e < n * n; e += nth) {
                const int i = e / n, j = e - i * n;
                double acc = i == j ? 1.0 : 0.0;
                for (int k = 0; k < n; ++k) acc += dare_lo(GH, ld, i, k) * dare_up(GH, ld, k, j);
                W1[i * ld + j] = acc;
                W2[i * ld + j] = i == j ? 1.0 : 0.0;
            }
            __syncthreads();
            if (!dare_gj(W1, ld, W2, ld, n, n, g, prow, krow)) {   // W2 = W^-1
                if (tid == 0) s_state = TREPB_DARE_SINGULAR;
                __syncthreads();
                break;
            }
            // W1 <- Z = W^-1 G (lower), Y = H W^-1 (upper)
            for (int e = tid; e < n * n; e += nth) {
                const int i = e / n, j = e - i * n;
                if (j <= i) {
                    double acc = 0.0;
                    for (int k = 0; k < n; ++k) acc += W2[i * ld + k] * dare_lo(GH, ld, k, j);
                    W1[i * ld + j] = acc;
                }
                if (j >= i) {
                    double acc = 0.0;
                    for (int k = 0; k < n; ++k) acc += dare_up(GH, ld, i, k) * W2[k * ld + j];
                    W1[i * ld + j + 1] = acc;
                }
            }
            __syncthreads();
            // one warp per row: W2 <- X = W^-1 A;  G += A Z A^T, H += A^T Y A (the change of H and H itself summed up)
            double d2 = 0.0, h2 = 0.0;
            for (int i = warp; i < n; i += nw) {
                for (int k = lane; k < n; k += 32) rb[k] = W2[i * ld + k];
                __syncwarp();
                for (int j = lane; j < n; j += 32) {
                    double acc = 0.0;
                    for (int k = 0; k < n; ++k) acc += rb[k] * Ab[k * ld + j];
                    W2[i * ld + j] = acc;
                }
                __syncwarp();
                for (int k = lane; k < n; k += 32) {   // (A Z)[i][k]
                    double acc = 0.0;
                    for (int q = 0; q < n; ++q) acc += Ab[i * ld + q] * dare_lo(W1, ld, q, k);
                    rb[k] = acc;
                }
                __syncwarp();
                for (int j = lane; j <= i; j += 32) {
                    double acc = 0.0;
                    for (int q = 0; q < n; ++q) acc += rb[q] * Ab[j * ld + q];
                    GH[i * ld + j] += acc;
                }
                __syncwarp();
                for (int k = lane; k < n; k += 32) {   // (A^T Y)[i][k]
                    double acc = 0.0;
                    for (int q = 0; q < n; ++q) acc += Ab[q * ld + i] * dare_up(W1, ld, q, k);
                    rb[k] = acc;
                }
                __syncwarp();
                for (int j = i + lane; j < n; j += 32) {
                    double acc = 0.0;
                    for (int q = 0; q < n; ++q) acc += rb[q] * Ab[q * ld + j];
                    const double h0 = GH[i * ld + j + 1], h1 = h0 + acc, dh = h1 - h0, w = j == i ? 1.0 : 2.0;
                    GH[i * ld + j + 1] = h1;
                    d2 += w * (dh * dh);
                    h2 += w * (h1 * h1);
                }
                __syncwarp();
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                d2 += __shfl_xor_sync(0xffffffffu, d2, o);
                h2 += __shfl_xor_sync(0xffffffffu, h2, o);
            }
            if (lane == 0) { red[warp] = d2; red[nw + warp] = h2; }
            __syncthreads();
            // one warp per row: A <- A X
            for (int i = warp; i < n; i += nw) {
                for (int k = lane; k < n; k += 32) rb[k] = Ab[i * ld + k];
                __syncwarp();
                for (int j = lane; j < n; j += 32) {
                    double acc = 0.0;
                    for (int k = 0; k < n; ++k) acc += rb[k] * W2[k * ld + j];
                    Ab[i * ld + j] = acc;
                }
                __syncwarp();
            }
            if (tid == 0) {
                double dn = 0.0, hn = 0.0;
                for (int w = 0; w < nw; ++w) { dn += red[w]; hn += red[nw + w]; }
                if (!(dn <= 1.7976931348623157e308 && hn <= 1.7976931348623157e308)) s_state = TREPB_DARE_NONFINITE;
                else if (dn <= p.tol * p.tol * hn) s_state = 1;
                else if (it >= p.max_it) s_state = TREPB_DARE_NOT_CONVERGED;
            }
            __syncthreads();
        }
        // ---- P = H, K = (R + B^T P B)^-1 (B^T P A + S^T) with the caller's A, B, R, S ----------------------------
        if (s_state == 1) {
            double* Bk = W1;                 // [n][m]
            double* PB = Bk + n * m;         // [n][m]
            double* M = PB + n * m;          // [m][m + n] = [R + B^T P B | B^T P A + S^T]
            const int ldm = m + n;
            double* Kp = M + m * ldm;        // [m][n] B^T P A + S^T, kept for the residual
            for (int e = tid; e < n * n; e += nth) {
                const int i = e / n, j = e - i * n;
                Ab[i * ld + j] = Ar[e];
                if (p.P) p.P[r * n * n + e] = dare_up(GH, ld, i, j);
            }
            for (int e = tid; e < n * m; e += nth) Bk[e] = Br[e];
            __syncthreads();
            for (int e = tid; e < n * m; e += nth) {
                const int i = e / m, c = e - i * m;
                double acc = 0.0;
                for (int k = 0; k < n; ++k) acc += dare_up(GH, ld, i, k) * Bk[k * m + c];
                PB[e] = acc;
            }
            __syncthreads();
            for (int e = tid; e < m * ldm; e += nth) {
                const int c = e / ldm, j = e - c * ldm;
                double acc = 0.0;
                if (j < m) {
                    for (int i = 0; i < n; ++i) acc += Bk[i * m + c] * PB[i * m + j];
                    acc += Rr[c * m + j];
                } else {
                    const int x = j - m;
                    for (int i = 0; i < n; ++i) acc += PB[i * m + c] * Ab[i * ld + x];
                    if (Sr) acc += Sr[x * m + c];
                    Kp[c * n + x] = acc;
                }
                M[e] = acc;
            }
            __syncthreads();
            if (!dare_gj(M, ldm, M + m, ldm, m, n, g, prow, krow)) {
                if (tid == 0) s_state = TREPB_DARE_SINGULAR;
            } else {
                if (p.K)
                    for (int e = tid; e < m * n; e += nth) {
                        const int c = e / n, x = e - c * n;
                        p.K[r * m * n + e] = M[c * ldm + m + x];
                    }
                // Without a stabilizing solution H grows without bound, and W = I + G H can lose so much accuracy
                // before anything overflows that the doubling stalls on a matrix that is no solution at all.  So the
                // answer is checked against the equation itself: ||A^T P A - P - Kp^T K + Q||_F <= 1e-6 times the
                // Frobenius norm of the four terms side by side (a converged P is some 1e-15 of it, a stalled one
                // O(1)), one warp per row.
                double r2 = 0.0, t2 = 0.0;
                for (int i = warp; i < n; i += nw) {
                    for (int k = lane; k < n; k += 32) {   // (A^T P)[i][k]
                        double acc = 0.0;
                        for (int q = 0; q < n; ++q) acc += Ab[q * ld + i] * dare_up(GH, ld, q, k);
                        rb[k] = acc;
                    }
                    __syncwarp();
                    for (int j = lane; j < n; j += 32) {
                        double apa = 0.0, kk = 0.0;
                        for (int k = 0; k < n; ++k) apa += rb[k] * Ab[k * ld + j];
                        for (int c = 0; c < m; ++c) kk += Kp[c * n + i] * M[c * ldm + m + j];
                        const double pij = dare_up(GH, ld, i, j), qij = 0.5 * (Qr[i * n + j] + Qr[j * n + i]);
                        const double v = apa - pij - kk + qij;
                        r2 += v * v;
                        t2 += apa * apa + pij * pij + kk * kk + qij * qij;
                    }
                    __syncwarp();
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    r2 += __shfl_xor_sync(0xffffffffu, r2, o);
                    t2 += __shfl_xor_sync(0xffffffffu, t2, o);
                }
                if (lane == 0) { red[warp] = r2; red[nw + warp] = t2; }
                __syncthreads();
                if (tid == 0) {
                    double rn = 0.0, tn = 0.0;
                    for (int w = 0; w < nw; ++w) { rn += red[w]; tn += red[nw + w]; }
                    if (!(rn <= 1.7976931348623157e308 && tn <= 1.7976931348623157e308)) s_state = TREPB_DARE_NONFINITE;
                    else if (!(rn <= 1e-12 * tn)) s_state = TREPB_DARE_NOT_CONVERGED;
                }
            }
            __syncthreads();
        }
        if (tid == 0) {
            p.status[r] = s_state == 1 ? TREPB_DARE_OK : s_state;
            if (p.iters) p.iters[r] = it;
        }
        __syncthreads();
    }
}

}  // namespace
}  // namespace trepb
