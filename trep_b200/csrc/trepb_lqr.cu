// Time-varying discrete LQR on the device: trep.discopt.dlqr.solve_tv_lqr (trep/discopt/dlqr.py:9-38),
// the backward Riccati sweep behind DSystem.calc_feedback_controller (trep/discopt/dsystem.py:474-494):
//
//     P = Q(K)
//     for k = K-1 .. 0:   gamma = R(k) + B^T P B ;  Kp = B^T P A ;  K[k] = gamma^-1 Kp
//                         P = Q(k) + A^T P A - Kp^T K[k] ;  P = (P + P^T) / 2
//
// One CTA per rollout (the sweep is sequential in k, rollouts are independent), P, P A and A[k] in
// shared memory (3 x nX^2 doubles: 154 KB for the marionette's nX = 80), A[k] / B[k] streamed from the
// slabs the linearize kernel wrote, so the linearization never leaves the GPU; K[k] goes straight into
// the layout trepb_project_batch reads (per-rollout gains).  Every product has the form
// C = X^T Y with both operands read along rows (P is symmetric): on the FP64 tensor cores
// (mma.sync m8n8k4, one warp per 16 x 40 tile, ragged edges read as zero) for nX >= 32, on 4 x 4 register
// tiles per thread below that; K[k] = gamma^-1 Kp (and the affine term) by a Gauss-Jordan elimination of
// [gamma | Kp | c] shared by the whole CTA; A[k-1], B[k-1] and Q(k) are fetched with cp.async while the
// current step is still multiplying.  One CTA of 16 warps per SM at the marionette's size, several smaller
// CTAs per SM for small states.
#include <cuda_runtime.h>
#include "trepb_nvtx.h"
#include <stdlib.h>
#include <string>
#include "../../include/trepb.h"
#include "trepb_coop_math.cuh"
#include "trepb_err.h"
#include "trepb_sweep.cuh"
#include "trepb_track.cuh"
#include "trepb_dare.cuh"
#include "trepb_dlyap.cuh"

namespace trepb {
namespace {

struct LqrParams {
    long long batch;
    int K, nX, nU;
    const double *A, *B, *Q, *R;
    int q_per_step, r_per_step;
    double *Kfb, *P0;
    int* status;
    // affine-quadratic extension (solve_tv_lq, dlqr.py:41-81); all null / zero for the plain LQR
    const double *S, *qv, *rv;         // cross term [K][nX][nU] (may be null), linear costs [K+1][nX], [K][nU]
    long long Qs, Rs, Ss, qs, rs;      // per-rollout strides of Q, R, S, q, r (0: shared by the batch)
    double *C, *b0;                    // [batch][K][nU], [batch][nX]
};

// C[i][j] (op)= sum_m Xt[m][i] * Y[m][j]   for i < M, j < N, m < Kd ; 4 x 4 tiles over the CTA.
//   mode 0: C = acc   1: C += acc   2: C -= acc
// VEC: ldx, ldy even and both operands 16-byte aligned -> the four operand values of a tile row come
// in as two 128-bit shared-memory loads each.
template <bool VEC>
__device__ __forceinline__ void gemm_tn(double* C, int ldc, const double* Xt, int ldx, const double* Y, int ldy,
                                        int M, int N, int Kd, int mode, int t0 = 0, int nt = 0) {
    // threads t0 .. t0+nt-1 of the CTA share the tiles (default: the whole CTA)
    if (nt == 0) nt = blockDim.x;
    const int me = (int)threadIdx.x - t0;
    if (me < 0 || me >= nt) return;
    const int ti = (M + 3) / 4, tj = (N + 3) / 4;
    for (int tile = me; tile < ti * tj; tile += nt) {
        const int i0 = (tile / tj) * 4, j0 = (tile % tj) * 4;
        double acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
        const bool full = i0 + 4 <= M && j0 + 4 <= N;
        if (full) {
            const double* xp = Xt + i0;
            const double* yp = Y + j0;
#pragma unroll 4
            for (int m = 0; m < Kd; ++m) {
                double x[4], y[4];
                if (VEC) {
                    const double2 x01 = *reinterpret_cast<const double2*>(xp), x23 = *reinterpret_cast<const double2*>(xp + 2);
                    const double2 y01 = *reinterpret_cast<const double2*>(yp), y23 = *reinterpret_cast<const double2*>(yp + 2);
                    x[0] = x01.x; x[1] = x01.y; x[2] = x23.x; x[3] = x23.y;
                    y[0] = y01.x; y[1] = y01.y; y[2] = y23.x; y[3] = y23.y;
                } else {
#pragma unroll
                    for (int a = 0; a < 4; ++a) { x[a] = xp[a]; y[a] = yp[a]; }
                }
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b) acc[a][b] += x[a] * y[b];
                xp += ldx; yp += ldy;
            }
        } else {
            for (int m = 0; m < Kd; ++m) {
                double x[4], y[4];
#pragma unroll
                for (int a = 0; a < 4; ++a) {
                    x[a] = i0 + a < M ? Xt[m * ldx + i0 + a] : 0.0;
                    y[a] = j0 + a < N ? Y[m * ldy + j0 + a] : 0.0;
                }
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b) acc[a][b] += x[a] * y[b];
            }
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                if (i0 + a < M && j0 + b < N) {
                    double* c = C + (i0 + a) * ldc + j0 + b;
                    if (mode == 0) *c = acc[a][b];
                    else if (mode == 1) *c += acc[a][b];
                    else *c -= acc[a][b];
                }
            }
    }
}

// The same product on the FP64 tensor-core path: mma.sync.aligned.m8n8k4 (DMMA), one warp per tile of
// (8 TI) x (8 TJ) outputs, TI + TJ operand fragments loaded per TI x TJ instructions of 256 fused
// multiply-adds.  Fragment layout (g = lane / 4, tg = lane % 4): A[g][tg] = Xt[m0 + tg][i + g],
// B[tg][g] = Y[m0 + tg][j + g], C[g][2 tg + {0, 1}].  Rows / columns beyond M, N, Kd read as zero and are
// not stored, so any shape works (nU = 18 runs as 24).  Warps w0 .. w0+nw-1 of the CTA share the tiles.
template <int TI, int TJ>
__device__ __forceinline__ void gemm_tn_dmma(double* C, int ldc, const double* Xt, int ldx, const double* Y, int ldy,
                                             int M, int N, int Kd, int mode, int w0, int nw) {
    const int warp = (int)(threadIdx.x >> 5) - w0, lane = threadIdx.x & 31;
    if (warp < 0 || warp >= nw) return;
    const int g = lane >> 2, tg = lane & 3;
    const int tm = (M + 8 * TI - 1) / (8 * TI), tn = (N + 8 * TJ - 1) / (8 * TJ);
    for (int tile = warp; tile < tm * tn; tile += nw) {
        const int i0 = (tile / tn) * 8 * TI, j0 = (tile % tn) * 8 * TJ;
        double c[TI][TJ][2];
        bool xin[TI], yin[TJ];
#pragma unroll
        for (int a = 0; a < TI; ++a) xin[a] = i0 + 8 * a + g < M;
#pragma unroll
        for (int b = 0; b < TJ; ++b) yin[b] = j0 + 8 * b + g < N;
#pragma unroll
        for (int a = 0; a < TI; ++a)
#pragma unroll
            for (int b = 0; b < TJ; ++b) c[a][b][0] = c[a][b][1] = 0.0;
        const double* xp = Xt + tg * ldx + i0 + g;
        const double* yp = Y + tg * ldy + j0 + g;
        for (int m0 = 0; m0 < Kd; m0 += 4) {
            const bool in = m0 + tg < Kd;
            double x[TI], y[TJ];
#pragma unroll
            for (int a = 0; a < TI; ++a) x[a] = (in && xin[a]) ? xp[8 * a] : 0.0;
#pragma unroll
            for (int b = 0; b < TJ; ++b) y[b] = (in && yin[b]) ? yp[8 * b] : 0.0;
#pragma unroll
            for (int a = 0; a < TI; ++a)
#pragma unroll
                for (int b = 0; b < TJ; ++b)
                    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                                 : "+d"(c[a][b][0]), "+d"(c[a][b][1]) : "d"(x[a]), "d"(y[b]));
            xp += 4 * ldx; yp += 4 * ldy;
        }
#pragma unroll
        for (int a = 0; a < TI; ++a)
#pragma unroll
            for (int b = 0; b < TJ; ++b) {
                const int i = i0 + 8 * a + g, j = j0 + 8 * b + 2 * tg;
                if (i >= M) continue;
                double* cp = C + i * ldc + j;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    if (j + h >= N) continue;
                    if (mode == 0) cp[h] = c[a][b][h];
                    else if (mode == 1) cp[h] += c[a][b][h];
                    else cp[h] -= c[a][b][h];
                }
            }
    }
}

// global -> shared copy that does not pass through registers (cp.async): issued early, waited for late,
// so the next step's A[k], B[k] and Q(k) arrive while the current step is still multiplying
__device__ __forceinline__ void async_copy(double* dst, const double* src, int n) {
    const unsigned d0 = (unsigned)__cvta_generic_to_shared(dst);
    if ((((unsigned long long)src | (unsigned long long)d0) & 15ull) == 0ull && (n & 1) == 0) {
        for (int e = threadIdx.x; e < n / 2; e += blockDim.x)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d0 + 16u * e), "l"(src + 2 * e) : "memory");
    } else {
        for (int e = threadIdx.x; e < n; e += blockDim.x)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d0 + 8u * e), "l"(src + e) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}
__device__ __forceinline__ void async_wait() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// K = gamma^-1 [Kp | c] by Gauss-Jordan elimination with implicitly scaled partial pivoting, the whole CTA
// on one system M = [gamma | Kp | c] (n rows, nc columns, leading dimension ldt): its elements are dealt
// out to the threads (at most kGJ each; GjElems holds their offsets, computed once per kernel), every warp
// finds the pivot of step k on its own (lane = row, two max-reductions over the bit pattern of |a| scale,
// lowest row among equals), every element outside the pivot row and right of column k takes one fused
// multiply-add, one __syncthreads per step.  No row is moved: order[k] = pivot row of step k, the solution
// row k is row order[k] divided by its pivot.  (The sweep is sequential in k and this solve sits on its
// critical path: a one-warp LU plus one right-hand side per thread took 55 % of a Riccati step.)
// Returns false if a scaled pivot is <= tol.
constexpr int kGJ = 4;
struct GjElems {
    int off[kGJ];   // i * ldt + j, or -1
    int row[kGJ];   // i * ldt
    int col[kGJ];   // j
};
__device__ __forceinline__ GjElems gj_elems(int n, int nc, int ldt) {
    GjElems g;
#pragma unroll
    for (int q = 0; q < kGJ; ++q) {
        const int e = (int)threadIdx.x + q * (int)blockDim.x;
        const bool in = e < n * nc;
        const int i = in ? e / nc : 0, j = e - i * nc;
        g.off[q] = in ? i * ldt + j : -1;
        g.row[q] = i * ldt;
        g.col[q] = j;
    }
    return g;
}
__device__ __forceinline__ bool cta_gauss_jordan(double* M, int ldt, int n, const GjElems& g, double* scl, double* rd,
                                                 int* order, double tol) {
    const int tid = threadIdx.x, lane = tid & 31, nth = blockDim.x;
    for (int i = tid; i < n; i += nth) {
        double sm_ = -1.0;
        for (int j = 0; j < n; ++j) { const double a = fabs(M[i * ldt + j]); if (a > sm_) sm_ = a; }
        scl[i] = 1.0 / sm_;
    }
    __syncthreads();
    // rows already used as pivots: a bit mask every thread keeps for itself (all threads compute the same pivots);
    // a flag array in shared memory would be written by one warp while a slower one still searches this step's pivot
    unsigned long long used = 0ull;
    for (int k = 0; k < n; ++k) {
        // pivot of column k among the rows not used yet (every warp computes the same answer)
        double best = 0.0;
        int br = 0x7fffffff;
        for (int r = lane; r < n; r += 32) {
            double v = ((used >> r) & 1ull) ? 0.0 : fabs(M[r * ldt + k] * scl[r]);
            if (!(v == v)) v = 0.0;
            if (v > best) { best = v; br = r; }
        }
        const unsigned long long bits = (unsigned long long)__double_as_longlong(best);
        const unsigned hi = (unsigned)(bits >> 32), lo = (unsigned)bits;
        const unsigned mh = __reduce_max_sync(0xffffffffu, hi);
        const unsigned ml = __reduce_max_sync(0xffffffffu, hi == mh ? lo : 0u);
        const int pr = (int)__reduce_min_sync(0xffffffffu, (hi == mh && lo == ml) ? (unsigned)br : 0x7fffffffu);
        const double bestv = __longlong_as_double((long long)(((unsigned long long)mh << 32) | ml));
        if (!(bestv > tol)) return false;
        const double* prow = M + pr * ldt;
        const double rdk = 1.0 / prow[k];
#pragma unroll
        for (int q = 0; q < kGJ; ++q) {
            if (g.off[q] < 0 || g.row[q] == pr * ldt || g.col[q] <= k) continue;
            M[g.off[q]] -= M[g.row[q] + k] * (rdk * prow[g.col[q]]);
        }
        used |= 1ull << pr;
        if (tid == 0) { order[k] = pr; rd[k] = rdk; }
        __syncthreads();
    }
    return true;
}

template <bool VEC, bool MMA>
__global__ void __launch_bounds__(512, 1) lqr_kernel(const LqrParams p) {
    extern __shared__ __align__(16) double sm[];
    const int nX = p.nX, nU = p.nU, K = p.K;
    const int nct = nU + nX + 1, ldg = nct | 1;    // columns / (odd) leading dimension of M = [gamma | Kp | c]
    const GjElems gje = gj_elems(nU, nct, ldg);
    double* P = sm;                                // [nX][nX]
    double* T = P + nX * nX;                       // P A
    double* As = T + nX * nX;                      // A[k]
    double* Bs = As + nX * nX;                     // B[k]            [nX][nU]
    double* W = Bs + nX * nU;                      // P B [nX][nU]
    double* Kp = W + nX * nU;                      // Kp = B^T P A    [nU][nX]
    double* Rs = Kp + nU * nX;                     // R(k)            [nU][nU]
    double* G = Rs + ((nU * nU + 1) & ~1);         // M = [gamma | Kp | c] [nU][ldt], eliminated in place
    double* scl = G + ((nU * ldg + 1) & ~1);       // [nU]
    double* rd = scl + nU;                         // [nU]
    int* order = (int*)(rd + nU);                  // [nU] pivot row of every elimination step (+ nU ints of padding)
    double* Ks = (double*)(order + 2 * nU);        // K[k] [nU][nX]   (2 nU ints = nU doubles: stays 8-byte aligned)
    // affine part (solve_tv_lq): b [nX], A^T b [nX], g = B^T b [nU] (+ r(k): the last column of M)
    double* bv = Ks + nU * nX;
    double* ab = bv + nX;
    double* gv = ab + nX;
    const bool affine = p.qv != nullptr;
    __shared__ int s_fail;
    for (long r = blockIdx.x; r < p.batch; r += gridDim.x) {
        const double* Ar = p.A + r * (long)K * nX * nX;
        const double* Br = p.B + r * (long)K * nX * nU;
        const double* Qr = p.Q + r * p.Qs;
        const double* Rr = p.R + r * p.Rs;
        const double* Sr = p.S ? p.S + r * p.Ss : nullptr;
        const double* qr = affine ? p.qv + r * p.qs : nullptr;
        const double* rr = affine ? p.rv + r * p.rs : nullptr;
        double* Kr = p.Kfb + r * (long)K * nU * nX;
        if (threadIdx.x == 0) s_fail = 0;
        async_copy(P, Qr + (p.q_per_step ? (long)K * nX * nX : 0), nX * nX);     // P = Q(K)
        async_copy(As, Ar + (long)(K - 1) * nX * nX, nX * nX);
        async_copy(Bs, Br + (long)(K - 1) * nX * nU, nX * nU);
        async_copy(Rs, Rr + (p.r_per_step ? (long)(K - 1) * nU * nU : 0), nU * nU);
        if (affine) for (int c = threadIdx.x; c < nX; c += blockDim.x) bv[c] = qr[(long)K * nX + c];   // b = q[K]
        for (int k = K - 1; k >= 0; --k) {
            async_wait();                                          // A[k], B[k], R(k) (and P) have landed
            __syncthreads();
            if (affine) {
                // A^T b and g = B^T b with the old b (columns of A / B, one per thread)
                for (int c = threadIdx.x; c < nX + nU; c += blockDim.x) {
                    double acc = 0.0;
                    if (c < nX) { for (int m = 0; m < nX; ++m) acc += As[m * nX + c] * bv[m]; ab[c] = acc; }
                    else { const int i = c - nX; for (int m = 0; m < nX; ++m) acc += Bs[m * nU + i] * bv[m]; gv[i] = acc; }
                }
            }
            const int nwarps = blockDim.x >> 5;
            if (MMA) {
                // tensor-core schedule (16 warps): T = P A on warps 0-9 next to W = P B on warps 10-14
                gemm_tn_dmma<2, 5>(T, nX, P, nX, As, nX, nX, nX, nX, 0, 0, 10);
                gemm_tn_dmma<2, 3>(W, nU, P, nX, Bs, nU, nX, nU, nX, 0, 10, nwarps - 10);
            } else {
                gemm_tn<VEC>(T, nX, P, nX, As, nX, nX, nX, nX, 0);     // T = P A      (P symmetric: P^T = P)
                gemm_tn<VEC>(W, nU, P, nX, Bs, nU, nX, nU, nX, 0);     // W = P B
            }
            for (int e = threadIdx.x; e < nU * nU; e += blockDim.x) G[(e / nU) * ldg + e % nU] = Rs[e];
            __syncthreads();
            async_copy(P, Qr + (p.q_per_step ? (long)k * nX * nX : 0), nX * nX);   // P is dead: start P <- Q(k)
            // gamma = R + B^T P B and Kp = B^T P A (tensor cores: 3 + 6 warp tiles)
            if (MMA) {
                gemm_tn_dmma<1, 3>(G, ldg, Bs, nU, W, nU, nU, nU, nX, 1, 0, 3);
                gemm_tn_dmma<1, 5>(Kp, nX, Bs, nU, T, nX, nU, nX, nX, 0, 3, nwarps - 3);
            } else {
                gemm_tn<VEC>(G, ldg, Bs, nU, W, nU, nU, nU, nX, 1);
                gemm_tn<VEC>(Kp, nX, Bs, nU, T, nX, nU, nX, nX, 0);
            }
            async_wait();                                          // Q(k) is in P
            __syncthreads();
            // P += A^T (P A) next to the set-up of the solve: Kp += S(k)^T (cross term), W <- Kp, c = r(k) + B^T b
            if (MMA) gemm_tn_dmma<2, 5>(P, nX, As, nX, T, nX, nX, nX, nX, 1, 0, 10);
            else gemm_tn<VEC>(P, nX, As, nX, T, nX, nX, nX, nX, 1);
            for (int e = threadIdx.x; e < nU * nX; e += blockDim.x) {
                const int i = e / nX, c = e - i * nX;
                double v = Kp[e];
                if (Sr) { v += Sr[(long)k * nX * nU + c * nU + i]; Kp[e] = v; }
                G[i * ldg + nU + c] = v;
            }
            for (int i = threadIdx.x; i < nU; i += blockDim.x) {
                double c = 0.0;
                if (affine) { gv[i] += rr[(long)k * nU + i]; c = gv[i]; }   // gv = r + B^T b
                G[i * ldg + nU + nX] = c;
            }
            __syncthreads();
            // K[k] = gamma^-1 Kp and C[k] = gamma^-1 (r + B^T b)
            if (!cta_gauss_jordan(G, ldg, nU, gje, scl, rd, order, 1e-300)) {
                s_fail = 1;   // every thread takes this branch (the pivots are computed redundantly by every warp)
                break;
            }
            for (int e = threadIdx.x; e < nU * nX; e += blockDim.x) {
                const int i = e / nX;
                Ks[e] = G[order[i] * ldg + nU + (e - i * nX)] * rd[i];
            }
            if (affine) {
                double* Ck = p.C + (r * (long)K + k) * nU;
                for (int i = threadIdx.x; i < nU; i += blockDim.x) Ck[i] = G[order[i] * ldg + nU + nX] * rd[i];
            }
            __syncthreads();
            double* Kk = Kr + (long)k * nU * nX;
            for (int e = threadIdx.x; e < nU * nX; e += blockDim.x) Kk[e] = Ks[e];
            if (affine) {
                // b = q[k] - K^T r + (A^T - K^T B^T) b = q[k] + A^T b - K^T (r + B^T b)
                for (int c = threadIdx.x; c < nX; c += blockDim.x) {
                    double acc = qr[(long)k * nX + c] + ab[c];
                    for (int i = 0; i < nU; ++i) acc -= Ks[i * nX + c] * gv[i];
                    bv[c] = acc;
                }
            }
            if (k > 0) {                                           // A, B are dead: fetch the next step's
                async_copy(As, Ar + (long)(k - 1) * nX * nX, nX * nX);
                async_copy(Bs, Br + (long)(k - 1) * nX * nU, nX * nU);
                if (p.r_per_step) async_copy(Rs, Rr + (long)(k - 1) * nU * nU, nU * nU);
            }
            if (MMA) gemm_tn_dmma<2, 5>(P, nX, Kp, nX, Ks, nX, nX, nX, nU, 2, 0, nwarps);   // P -= Kp^T K[k]
            else gemm_tn<VEC>(P, nX, Kp, nX, Ks, nX, nX, nX, nU, 2);
            __syncthreads();
            // P = (P + P^T) / 2, one off-diagonal per warp pass: (i, i + d) and its mirror are both read with
            // stride nX + 1 (a row-by-row sweep reads the mirror with stride nX: a 32-way bank conflict at nX = 80)
            for (int d = 1 + (int)(threadIdx.x >> 5); d < nX; d += nwarps) {
                for (int i = threadIdx.x & 31; i + d < nX; i += 32) {
                    const int a = i * nX + i + d, b = (i + d) * nX + i;
                    const double v = (P[a] + P[b]) / 2.0;
                    P[a] = v;
                    P[b] = v;
                }
            }
        }
        async_wait();
        __syncthreads();
        if (p.P0) {
            double* Pr = p.P0 + r * (long)nX * nX;
            for (int e = threadIdx.x; e < nX * nX; e += blockDim.x) Pr[e] = P[e];
        }
        if (affine && p.b0) for (int c = threadIdx.x; c < nX; c += blockDim.x) p.b0[r * (long)nX + c] = bv[c];
        if (threadIdx.x == 0) p.status[r] = s_fail ? ST_SINGULAR : ST_OK;
        __syncthreads();
    }
}

int lqr_fail(int code, const std::string& m) { last_error() = m; return code; }

}  // namespace
}  // namespace trepb

using namespace trepb;

namespace {
// CUDA events around the last Riccati launch of each device (trepb_lqr_last_kernel_ms)
struct LqrTimer {
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool ok = false;
};
LqrTimer& lqr_timer(int device) {
    static LqrTimer t[64];
    LqrTimer& x = t[device & 63];
    if (!x.ok) x.ok = cudaEventCreate(&x.e0) == cudaSuccess && cudaEventCreate(&x.e1) == cudaSuccess;
    return x;
}

int lqr_launch(int device, LqrParams& p, cudaStream_t stream) {
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    const int nX = p.nX, nU = p.nU, ldg = (nU + nX + 1) | 1;
    const size_t doubles = 3 * (size_t)nX * nX + 4 * (size_t)nX * nU + (size_t)nU * nU + (size_t)nU * ldg + 4 * (size_t)nU + 16
                           + 2 * (size_t)nX + 2 * (size_t)nU + 2;
    const size_t smem = doubles * sizeof(double);
    int smem_optin = 0, sms = 0;
    e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    if (smem > (size_t)smem_optin)
        return lqr_fail(TREPB_ERR_UNSUPPORTED, "state dimension too large for the shared-memory Riccati sweep");
    const bool vec = nX % 2 == 0 && nU % 2 == 0;   // every operand block then starts 16-byte aligned with an even row length
    // tensor-core schedule for states large enough to fill its warp tiles (TREPB_LQR_NO_MMA=1: scalar tiles, for comparison)
    const char* no_mma = getenv("TREPB_LQR_NO_MMA");
    const bool mma = nX >= 32 && !(no_mma && no_mma[0] == '1');
    const void* fn = mma ? (vec ? (const void*)lqr_kernel<true, true> : (const void*)lqr_kernel<false, true>) : vec ? (const void*)lqr_kernel<true, false> : (const void*)lqr_kernel<false, false>;
    e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    const int tiles = ((nX + 3) / 4) * ((nX + 3) / 4);
    int block = ((tiles + 31) / 32) * 32;
    if (block > 512) block = 512;
    if (block < 64) block = 64;
    if (mma) block = 512;   // the tensor-core schedule assigns products to warps 0-9 and 10-14
    // the elimination deals the nU x (nU + nX + 1) elements of [gamma | Kp | c] out to the threads, at most 4 each
    // the limit below already refuses every nU >= 45; this one is what makes cta_gauss_jordan's 64-bit `used` mask safe
    if (nU > 64) return lqr_fail(TREPB_ERR_UNSUPPORTED, "more than 64 inputs");
    while (block < 512 && (long long)nU * (nU + nX + 1) > 4LL * block) block += 32;
    if ((long long)nU * (nU + nX + 1) > 4LL * block)
        return lqr_fail(TREPB_ERR_UNSUPPORTED, "input dimension too large for the in-kernel gamma solve");
    // small systems: as many CTAs per SM as registers / shared memory allow (one rollout per CTA)
    int occ = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, block, smem) != cudaSuccess || occ < 1) occ = 1;
    const long long slots = (long long)sms * occ;
    const long long grid = p.batch < slots ? p.batch : slots;
    LqrTimer& tm = lqr_timer(device);
    if (tm.ok) cudaEventRecord(tm.e0, stream);
    if (mma && vec) lqr_kernel<true, true><<<(int)grid, block, smem, stream>>>(p);
    else if (mma) lqr_kernel<false, true><<<(int)grid, block, smem, stream>>>(p);
    else if (vec) lqr_kernel<true, false><<<(int)grid, block, smem, stream>>>(p);
    else lqr_kernel<false, false><<<(int)grid, block, smem, stream>>>(p);
    if (tm.ok) cudaEventRecord(tm.e1, stream);
    e = cudaGetLastError();
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    return TREPB_OK;
}
}  // namespace

extern "C" int trepb_lqr_last_kernel_ms(int device, float* ms) {
    if (!ms) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    LqrTimer& tm = lqr_timer(device);
    if (!tm.ok) return lqr_fail(TREPB_ERR_CUDA, "no events");
    e = cudaEventSynchronize(tm.e1);
    if (e == cudaSuccess) e = cudaEventElapsedTime(ms, tm.e0, tm.e1);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    return TREPB_OK;
}

extern "C" int trepb_lqr_batch_dev(int device, const trepb_lqr_args* a, void* stream) {
    TREPB_NVTX("trepb_lqr_batch_dev");
    if (!a) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    if (a->batch < 0 || a->nsteps < 1 || a->nX < 1 || a->nU < 1) return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    if (!a->A || !a->B || !a->Q || !a->R || !a->Kfb || !a->status) return lqr_fail(TREPB_ERR_INVALID, "A, B, Q, R, Kfb and status are required");
    if (a->batch == 0) return TREPB_OK;
    LqrParams p{};
    p.batch = a->batch; p.K = a->nsteps; p.nX = a->nX; p.nU = a->nU;
    p.A = a->A; p.B = a->B; p.Q = a->Q; p.R = a->R; p.q_per_step = a->q_per_step; p.r_per_step = a->r_per_step;
    p.Kfb = a->Kfb; p.P0 = a->P0; p.status = a->status;
    return lqr_launch(device, p, (cudaStream_t)stream);
}

extern "C" int trepb_lq_batch_dev(int device, const trepb_lq_args* a, void* stream) {
    TREPB_NVTX("trepb_lq_batch_dev");
    if (!a) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    if (a->batch < 0 || a->nsteps < 1 || a->nX < 1 || a->nU < 1) return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    if (!a->A || !a->B || !a->Q || !a->R || !a->q || !a->r || !a->Kfb || !a->C || !a->status)
        return lqr_fail(TREPB_ERR_INVALID, "A, B, Q, R, q, r, Kfb, C and status are required");
    if (a->batch == 0) return TREPB_OK;
    const long long K = a->nsteps, nX = a->nX, nU = a->nU, per = a->cost_per_rollout ? 1 : 0;
    LqrParams p{};
    p.batch = a->batch; p.K = a->nsteps; p.nX = a->nX; p.nU = a->nU;
    p.A = a->A; p.B = a->B; p.Q = a->Q; p.R = a->R; p.q_per_step = 1; p.r_per_step = 1;
    p.S = a->S; p.qv = a->q; p.rv = a->r;
    p.Qs = per * (K + 1) * nX * nX; p.Rs = per * K * nU * nU; p.Ss = per * K * nX * nU;
    p.qs = per * (K + 1) * nX; p.rs = per * K * nU;
    p.Kfb = a->Kfb; p.C = a->C; p.P0 = a->P0; p.b0 = a->b0; p.status = a->status;
    return lqr_launch(device, p, (cudaStream_t)stream);
}

extern "C" int trepb_lq_batch(int device, const trepb_lq_args* a) {
    TREPB_NVTX("trepb_lq_batch");
    if (!a) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    if (a->batch < 0 || a->nsteps < 1 || a->nX < 1 || a->nU < 1) return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    if (!a->A || !a->B || !a->Q || !a->R || !a->q || !a->r || !a->Kfb || !a->C || !a->status)
        return lqr_fail(TREPB_ERR_INVALID, "A, B, Q, R, q, r, Kfb, C and status are required");
    if (a->batch == 0) return TREPB_OK;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    const size_t Rn = (size_t)a->batch, K = (size_t)a->nsteps, nX = (size_t)a->nX, nU = (size_t)a->nU;
    const size_t cm = a->cost_per_rollout ? Rn : 1;
    // host -> device staging: {source, bytes} in, {destination, bytes} out
    const void* in_src[7] = {a->A, a->B, a->Q, a->R, a->S, a->q, a->r};
    const size_t in_n[7] = {Rn * K * nX * nX, Rn * K * nX * nU, cm * (K + 1) * nX * nX, cm * K * nU * nU,
                            a->S ? cm * K * nX * nU : 0, cm * (K + 1) * nX, cm * K * nU};
    void* out_dst[4] = {a->Kfb, a->C, a->P0, a->b0};
    const size_t out_n[4] = {Rn * K * nU * nX, Rn * K * nU, a->P0 ? Rn * nX * nX : 0, a->b0 ? Rn * nX : 0};
    double* din[7] = {nullptr}; double* dout[4] = {nullptr};
    int* dS = nullptr;
    int rc = TREPB_OK;
#define LQ(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess && rc == TREPB_OK) rc = lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e_)); } while (0)
    for (int i = 0; i < 7; ++i) if (in_n[i]) { LQ(cudaMalloc(&din[i], in_n[i] * 8)); if (rc == TREPB_OK) LQ(cudaMemcpy(din[i], in_src[i], in_n[i] * 8, cudaMemcpyHostToDevice)); }
    for (int i = 0; i < 4; ++i) if (out_n[i]) LQ(cudaMalloc(&dout[i], out_n[i] * 8));
    LQ(cudaMalloc(&dS, (Rn ? Rn : 1) * 4));
    if (rc == TREPB_OK && Rn) {
        trepb_lq_args d = *a;
        d.A = din[0]; d.B = din[1]; d.Q = din[2]; d.R = din[3]; d.S = din[4]; d.q = din[5]; d.r = din[6];
        d.Kfb = dout[0]; d.C = dout[1]; d.P0 = dout[2]; d.b0 = dout[3]; d.status = dS;
        rc = trepb_lq_batch_dev(device, &d, nullptr);
    }
    if (rc == TREPB_OK) {
        for (int i = 0; i < 4; ++i) if (out_n[i]) LQ(cudaMemcpy(out_dst[i], dout[i], out_n[i] * 8, cudaMemcpyDeviceToHost));
        if (Rn) LQ(cudaMemcpy(a->status, dS, Rn * 4, cudaMemcpyDeviceToHost));
    }
#undef LQ
    for (int i = 0; i < 7; ++i) cudaFree(din[i]);
    for (int i = 0; i < 4; ++i) cudaFree(dout[i]);
    cudaFree(dS);
    return rc;
}

extern "C" int trepb_lqr_batch(int device, const trepb_lqr_args* a) {
    TREPB_NVTX("trepb_lqr_batch");
    if (!a) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    if (a->batch < 0 || a->nsteps < 1 || a->nX < 1 || a->nU < 1) return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    if (a->batch == 0) return TREPB_OK;
    if (!a->A || !a->B || !a->Q || !a->R || !a->Kfb || !a->status) return lqr_fail(TREPB_ERR_INVALID, "A, B, Q, R, Kfb and status are required");
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    const size_t R = (size_t)a->batch, K = (size_t)a->nsteps, nX = (size_t)a->nX, nU = (size_t)a->nU;
    const size_t nA = R * K * nX * nX, nB = R * K * nX * nU, nQ = (a->q_per_step ? K + 1 : 1) * nX * nX,
                 nR = (a->r_per_step ? K : 1) * nU * nU, nK = R * K * nU * nX, nP = R * nX * nX;
    double *dA = nullptr, *dB = nullptr, *dQ = nullptr, *dR = nullptr, *dK = nullptr, *dP = nullptr;
    int* dS = nullptr;
    int rc = TREPB_OK;
#define LQ(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess && rc == TREPB_OK) rc = lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e_)); } while (0)
    LQ(cudaMalloc(&dA, nA * 8)); LQ(cudaMalloc(&dB, nB * 8)); LQ(cudaMalloc(&dQ, nQ * 8)); LQ(cudaMalloc(&dR, nR * 8));
    LQ(cudaMalloc(&dK, nK * 8)); LQ(cudaMalloc(&dP, nP * 8)); LQ(cudaMalloc(&dS, (R ? R : 1) * 4));
    if (rc == TREPB_OK) {
        LQ(cudaMemcpy(dA, a->A, nA * 8, cudaMemcpyHostToDevice)); LQ(cudaMemcpy(dB, a->B, nB * 8, cudaMemcpyHostToDevice));
        LQ(cudaMemcpy(dQ, a->Q, nQ * 8, cudaMemcpyHostToDevice)); LQ(cudaMemcpy(dR, a->R, nR * 8, cudaMemcpyHostToDevice));
    }
    if (rc == TREPB_OK) {
        trepb_lqr_args d = *a;
        d.A = dA; d.B = dB; d.Q = dQ; d.R = dR; d.Kfb = dK; d.P0 = a->P0 ? dP : nullptr; d.status = dS;
        rc = trepb_lqr_batch_dev(device, &d, nullptr);
    }
    if (rc == TREPB_OK) {
        LQ(cudaMemcpy(a->Kfb, dK, nK * 8, cudaMemcpyDeviceToHost));
        if (a->P0) LQ(cudaMemcpy(a->P0, dP, nP * 8, cudaMemcpyDeviceToHost));
        LQ(cudaMemcpy(a->status, dS, R * 4, cudaMemcpyDeviceToHost));
    }
#undef LQ
    cudaFree(dA); cudaFree(dB); cudaFree(dQ); cudaFree(dR); cudaFree(dK); cudaFree(dP); cudaFree(dS);
    return rc;
}

// ---- tangent / adjoint sweeps (trepb_sweep.cuh) ----------------------------------------------------------------
namespace {
int sweep_launch(int device, SweepParams& p, bool tangent, cudaStream_t stream) {
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    // one team of lanes per rollout, a power of two covering the longer of a state row / an input row
    const int rows = p.nX > p.nU ? p.nX : p.nU;
    int team = 1;
    while (team < rows && team < 128) team <<= 1;   // rows beyond 128 are strided over the team
    const int block = team < 64 ? 64 : team, teams = block / team;
    int smem_optin = 0;
    e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    // the deepest ring that fits: small states prefetch 7 steps ahead, the marionette's 74 KB steps one
    int stages = 8;
    while (stages >= 2 && (size_t)teams * sweep_team_doubles(p.nX, p.nU, stages) * 8 > (size_t)smem_optin) stages /= 2;
    if (stages < 2) return lqr_fail(TREPB_ERR_UNSUPPORTED, "state dimension too large for the shared-memory sweep");
    const size_t smem = (size_t)teams * sweep_team_doubles(p.nX, p.nU, stages) * 8;
    p.team = team; p.stages = stages;
    const void* fn = tangent ? (const void*)sweep_kernel<true> : (const void*)sweep_kernel<false>;
    e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    long long grid = (p.batch + teams - 1) / teams;
    if (grid > (1LL << 24)) grid = 1LL << 24;   // the kernel strides over the rest
    if (tangent) sweep_kernel<true><<<(unsigned)grid, block, smem, stream>>>(p);
    else sweep_kernel<false><<<(unsigned)grid, block, smem, stream>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    return TREPB_OK;
}

// the checks every tangent / adjoint entry point makes before any CUDA call; -1 = go on
int tangent_check(const trepb_tangent_args* a) {
    if (!a) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    if (a->batch < 0 || a->nsteps < 1 || a->nX < 1 || a->nU < 0) return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    if (!a->A || !a->dX || (a->nU > 0 && (!a->B || !a->K || !a->dU)))
        return lqr_fail(TREPB_ERR_INVALID, "A and dX are required, and B, K and dU when nU > 0");
    if (a->batch == 0) return TREPB_OK;
    return -1;
}
int adjoint_check(const trepb_adjoint_args* a) {
    if (!a) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    if (a->batch < 0 || a->nsteps < 1 || a->nX < 1 || a->nU < 0) return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    if (!a->A || !a->m_dx || !a->z || (a->K && a->nU > 0 && !a->B))
        return lqr_fail(TREPB_ERR_INVALID, "A, m_dx and z are required, and B when K is given");
    if (a->batch == 0) return TREPB_OK;
    return -1;
}

// host -> device staging of n_in inputs and n_out outputs around `run(device pointers)` (null / empty arrays
// stay null); synchronous, like trepb_lq_batch
template <int NI, int NO, class Run>
int sweep_staged(int device, const void* const (&src)[NI], const size_t (&in_n)[NI], void* const (&dst)[NO],
                 const size_t (&out_n)[NO], Run run) {
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    double* din[NI] = {nullptr};
    double* dout[NO] = {nullptr};
    int rc = TREPB_OK;
#define SW(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess && rc == TREPB_OK) rc = lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e_)); } while (0)
    for (int i = 0; i < NI; ++i)
        if (src[i] && in_n[i]) {
            SW(cudaMalloc(&din[i], in_n[i] * 8));
            if (rc == TREPB_OK) SW(cudaMemcpy(din[i], src[i], in_n[i] * 8, cudaMemcpyHostToDevice));
        }
    for (int i = 0; i < NO; ++i) if (dst[i] && out_n[i]) SW(cudaMalloc(&dout[i], out_n[i] * 8));
    if (rc == TREPB_OK) rc = run(din, dout);
    if (rc == TREPB_OK) SW(cudaStreamSynchronize(nullptr));
    if (rc == TREPB_OK)
        for (int i = 0; i < NO; ++i) if (dout[i]) SW(cudaMemcpy(dst[i], dout[i], out_n[i] * 8, cudaMemcpyDeviceToHost));
#undef SW
    for (int i = 0; i < NI; ++i) cudaFree(din[i]);
    for (int i = 0; i < NO; ++i) cudaFree(dout[i]);
    return rc;
}
}  // namespace

extern "C" int trepb_tangent_batch_dev(int device, const trepb_tangent_args* a, void* stream) {
    TREPB_NVTX("trepb_tangent_batch_dev");
    const int c = tangent_check(a);
    if (c >= 0) return c;
    SweepParams p{};
    p.batch = a->batch; p.K = a->nsteps; p.nX = a->nX; p.nU = a->nU;
    p.A = a->A; p.B = a->nU ? a->B : nullptr; p.Kfb = a->nU ? a->K : nullptr;
    p.vx = a->bdX; p.vu = a->nU ? a->bdU : nullptr; p.x0 = a->x0;
    p.ox = a->dX; p.ou = a->nU ? a->dU : nullptr;
    return sweep_launch(device, p, true, (cudaStream_t)stream);
}

extern "C" int trepb_adjoint_batch_dev(int device, const trepb_adjoint_args* a, void* stream) {
    TREPB_NVTX("trepb_adjoint_batch_dev");
    const int c = adjoint_check(a);
    if (c >= 0) return c;
    SweepParams p{};
    p.batch = a->batch; p.K = a->nsteps; p.nX = a->nX; p.nU = a->nU;
    p.A = a->A; p.B = a->nU && a->K ? a->B : nullptr; p.Kfb = a->nU ? a->K : nullptr;
    p.vx = a->l_dx; p.vu = a->nU && a->K ? a->l_du : nullptr; p.x0 = a->m_dx;
    p.ox = a->z; p.ou = a->z1;
    return sweep_launch(device, p, false, (cudaStream_t)stream);
}

extern "C" int trepb_tangent_batch(int device, const trepb_tangent_args* a) {
    TREPB_NVTX("trepb_tangent_batch");
    const int c = tangent_check(a);
    if (c >= 0) return c;
    const size_t Rn = (size_t)a->batch, K = (size_t)a->nsteps, nX = (size_t)a->nX, nU = (size_t)a->nU;
    const void* const src[6] = {a->A, a->B, a->K, a->bdX, a->bdU, a->x0};
    const size_t in_n[6] = {Rn * K * nX * nX, Rn * K * nX * nU, Rn * K * nU * nX, Rn * (K + 1) * nX, Rn * K * nU, Rn * nX};
    void* const dst[2] = {a->dX, a->dU};
    const size_t out_n[2] = {Rn * (K + 1) * nX, Rn * K * nU};
    return sweep_staged(device, src, in_n, dst, out_n, [&](double* const* d, double* const* o) {
        trepb_tangent_args x = *a;
        x.A = d[0]; x.B = d[1]; x.K = d[2]; x.bdX = d[3]; x.bdU = d[4]; x.x0 = d[5]; x.dX = o[0]; x.dU = o[1];
        return trepb_tangent_batch_dev(device, &x, nullptr);
    });
}

extern "C" int trepb_adjoint_batch(int device, const trepb_adjoint_args* a) {
    TREPB_NVTX("trepb_adjoint_batch");
    const int c = adjoint_check(a);
    if (c >= 0) return c;
    const size_t Rn = (size_t)a->batch, K = (size_t)a->nsteps, nX = (size_t)a->nX, nU = (size_t)a->nU;
    const void* const src[6] = {a->A, a->B, a->K, a->l_dx, a->l_du, a->m_dx};
    const size_t in_n[6] = {Rn * K * nX * nX, Rn * K * nX * nU, Rn * K * nU * nX, Rn * K * nX, Rn * K * nU, Rn * nX};
    void* const dst[2] = {a->z, a->z1};
    const size_t out_n[2] = {Rn * (K + 1) * nX, Rn * K * nX};
    return sweep_staged(device, src, in_n, dst, out_n, [&](double* const* d, double* const* o) {
        trepb_adjoint_args x = *a;
        x.A = d[0]; x.B = d[1]; x.K = d[2]; x.l_dx = d[3]; x.l_du = d[4]; x.m_dx = d[5]; x.z = o[0]; x.z1 = o[1];
        return trepb_adjoint_batch_dev(device, &x, nullptr);
    });
}

// ---- tracking cost, LQ model and line-search candidates (trepb_track.cuh) ----------------------------------------
namespace {
// the checks every track / candidates entry point makes before any CUDA call; -1 = go on
int track_check(const trepb_track_args* a) {
    if (!a) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    if (a->batch < 0 || a->nsteps < 1 || a->nX < 1 || a->nU < 0 || a->nref < 1) return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    const long long nX = a->nX, nU = a->nU, K = a->nsteps;
    if ((K + 1) * nX * nX + K * nX * nU + K * nU * nU > 0x7fffffffLL || (K + 1) * (nX + nU) > 0x7fffffffLL)
        return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    const bool grad = a->cost || a->dcost || a->q || a->r || a->l_dx || a->m_dx;
    const bool model = a->Qm || a->Sm || a->Rm;
    if (grad && (!a->X || !a->Xd || !a->Q || (nU > 0 && (!a->U || !a->Ud || !a->R))))
        return lqr_fail(TREPB_ERR_INVALID, "X, Xd and Q are required for the cost outputs, and U, Ud and R when nU > 0");
    if (a->dcost && (!a->dX || (nU > 0 && !a->dU))) return lqr_fail(TREPB_ERR_INVALID, "dcost needs dX and dU");
    const int newton = (a->fdxdx != nullptr) + (nU > 0 && a->fdxdu != nullptr) + (nU > 0 && a->fdudu != nullptr);
    if (newton != 0 && newton != (nU > 0 ? 3 : 1))
        return lqr_fail(TREPB_ERR_INVALID, "fdxdx, fdxdu and fdudu go together");
    if ((model || newton) && (!a->Qm || !a->Q || (nU > 0 && (!a->Rm || !a->R))))
        return lqr_fail(TREPB_ERR_INVALID, "the model needs Qm and Q, and Rm and R when nU > 0");
    if (a->batch == 0) return TREPB_OK;
    return -1;
}
int candidates_check(const trepb_candidates_args* a) {
    if (!a) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    if (a->groups < 0 || a->ncand < 1 || a->nsteps < 1 || a->nX < 1 || a->nU < 0 || a->nrollouts < 0)
        return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    const long long nX = a->nX, nU = a->nU, K = a->nsteps;
    if ((K + 1) * nX + K * nU + K * nU * nX > 0x7fffffffLL) return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    if (!a->lam || !a->X || !a->dX || !a->bX || (nU > 0 && (!a->U || !a->dU || !a->Kproj || !a->bU || !a->Kc)))
        return lqr_fail(TREPB_ERR_INVALID, "lam, X, dX and bX are required, and U, dU, Kproj, bU and Kc when nU > 0");
    if (a->groups == 0) return TREPB_OK;
    return -1;
}

// host -> device staging of inputs and outputs given in bytes around `run(device pointers)` (null / empty arrays
// stay null); synchronous, like the sweeps' host-pointer calls
template <int NI, int NO, class Run>
int stage_bytes(int device, const void* const (&src)[NI], const size_t (&in_b)[NI], void* const (&dst)[NO],
                const size_t (&out_b)[NO], Run run) {
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    void* din[NI] = {nullptr};
    void* dout[NO] = {nullptr};
    int rc = TREPB_OK;
#define SB(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess && rc == TREPB_OK) rc = lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e_)); } while (0)
    for (int i = 0; i < NI; ++i)
        if (src[i] && in_b[i]) {
            SB(cudaMalloc(&din[i], in_b[i]));
            if (rc == TREPB_OK) SB(cudaMemcpyAsync(din[i], src[i], in_b[i], cudaMemcpyHostToDevice, nullptr));
        }
    for (int i = 0; i < NO; ++i) if (dst[i] && out_b[i]) SB(cudaMalloc(&dout[i], out_b[i]));
    if (rc == TREPB_OK) rc = run(din, dout);
    if (rc == TREPB_OK)
        for (int i = 0; i < NO; ++i) if (dout[i]) SB(cudaMemcpyAsync(dst[i], dout[i], out_b[i], cudaMemcpyDeviceToHost, nullptr));
    SB(cudaStreamSynchronize(nullptr));
#undef SB
    for (int i = 0; i < NI; ++i) cudaFree(din[i]);
    for (int i = 0; i < NO; ++i) cudaFree(dout[i]);
    return rc;
}
}  // namespace

extern "C" int trepb_track_batch_dev(int device, const trepb_track_args* a, void* stream) {
    TREPB_NVTX("trepb_track_batch_dev");
    const int c = track_check(a);
    if (c >= 0) return c;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    TrackParams p{};
    const int nU = a->nU;
    p.batch = a->batch; p.K = a->nsteps; p.nX = a->nX; p.nU = nU;
    p.X = a->X; p.U = nU ? a->U : nullptr; p.Xd = a->Xd; p.Ud = nU ? a->Ud : nullptr; p.Q = a->Q; p.R = nU ? a->R : nullptr;
    p.ref = a->ref_index; p.dX = a->dX; p.dU = nU ? a->dU : nullptr;
    p.fxx = a->fdxdx; p.fxu = nU ? a->fdxdu : nullptr; p.fuu = nU ? a->fdudu : nullptr;
    p.cost = a->cost; p.dcost = a->dcost; p.q = a->q; p.r = nU ? a->r : nullptr; p.l_dx = a->l_dx; p.m_dx = a->m_dx;
    p.Qm = a->Qm; p.Sm = nU ? a->Sm : nullptr; p.Rm = nU ? a->Rm : nullptr;
    const bool grad = p.cost || p.dcost || p.q || p.r || p.l_dx || p.m_dx;
    const int block = 256;
    // cost role: one CTA per trajectory (strided beyond 2^20); a tile of about 2048 staged doubles per CTA
    const int cols = a->nX + nU;
    int tile = 2048 / cols;
    tile = tile < 1 ? 1 : tile > 256 ? 256 : tile;
    p.tile = tile;
    p.cost_blocks = grad ? (int)(p.batch < (1LL << 20) ? p.batch : (1LL << 20)) : 0;
    const size_t smem = grad ? (size_t)track_smem_doubles(a->nX, nU, tile) * 8 : 0;
    // model role: CTAs per trajectory such that each lane streams about four elements of the model
    long long model_blocks = 0;
    if (p.Qm) {
        const long long per = (p.K + 1LL) * a->nX * a->nX + (p.Sm ? (long long)p.K * a->nX * nU : 0) +
                              (p.Rm ? (long long)p.K * nU * nU : 0);
        p.model_bpt = (int)((per + 4LL * block - 1) / (4LL * block));
        model_blocks = p.batch * p.model_bpt;
        if (model_blocks > (1LL << 22)) model_blocks = 1LL << 22;
    }
    if (smem > 48 * 1024) {
        e = cudaFuncSetAttribute((const void*)track_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    }
    const long long grid = p.cost_blocks + model_blocks;
    if (grid == 0) return TREPB_OK;
    track_kernel<<<(unsigned)grid, block, smem, (cudaStream_t)stream>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    return TREPB_OK;
}

extern "C" int trepb_track_batch(int device, const trepb_track_args* a) {
    TREPB_NVTX("trepb_track_batch");
    const int c = track_check(a);
    if (c >= 0) return c;
    const size_t Rn = (size_t)a->batch, K = (size_t)a->nsteps, nX = (size_t)a->nX, nU = (size_t)a->nU, nr = (size_t)a->nref;
    const size_t d = 8;
    const void* const src[12] = {a->X, a->U, a->Xd, a->Ud, a->Q, a->R, a->ref_index, a->dX, a->dU,
                                 a->fdxdx, a->fdxdu, a->fdudu};
    const size_t in_b[12] = {Rn * (K + 1) * nX * d, Rn * K * nU * d, nr * (K + 1) * nX * d, nr * K * nU * d, nX * nX * d,
                             nU * nU * d, Rn * 4, Rn * (K + 1) * nX * d, Rn * K * nU * d, Rn * K * nX * nX * d,
                             Rn * K * nX * nU * d, Rn * K * nU * nU * d};
    void* const dst[9] = {a->cost, a->dcost, a->q, a->r, a->l_dx, a->m_dx, a->Qm, a->Sm, a->Rm};
    const size_t out_b[9] = {Rn * d, Rn * d, Rn * (K + 1) * nX * d, Rn * K * nU * d, Rn * K * nX * d, Rn * nX * d,
                             Rn * (K + 1) * nX * nX * d, Rn * K * nX * nU * d, Rn * K * nU * nU * d};
    return stage_bytes(device, src, in_b, dst, out_b, [&](void* const* i, void* const* o) {
        trepb_track_args x = *a;
        x.X = (const double*)i[0]; x.U = (const double*)i[1]; x.Xd = (const double*)i[2]; x.Ud = (const double*)i[3];
        x.Q = (const double*)i[4]; x.R = (const double*)i[5]; x.ref_index = (const int32_t*)i[6];
        x.dX = (const double*)i[7]; x.dU = (const double*)i[8]; x.fdxdx = (const double*)i[9];
        x.fdxdu = (const double*)i[10]; x.fdudu = (const double*)i[11];
        x.cost = (double*)o[0]; x.dcost = (double*)o[1]; x.q = (double*)o[2]; x.r = (double*)o[3];
        x.l_dx = (double*)o[4]; x.m_dx = (double*)o[5]; x.Qm = (double*)o[6]; x.Sm = (double*)o[7]; x.Rm = (double*)o[8];
        return trepb_track_batch_dev(device, &x, nullptr);
    });
}

extern "C" int trepb_candidates_batch_dev(int device, const trepb_candidates_args* a, void* stream) {
    TREPB_NVTX("trepb_candidates_batch_dev");
    const int c = candidates_check(a);
    if (c >= 0) return c;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    CandParams p{};
    const int nU = a->nU;
    p.G = a->groups; p.M = a->ncand; p.K = a->nsteps; p.nX = a->nX; p.nU = nU;
    p.rows = a->rows; p.lam = a->lam; p.X = a->X; p.U = nU ? a->U : nullptr; p.dX = a->dX; p.dU = nU ? a->dU : nullptr;
    p.Kp = nU ? a->Kproj : nullptr; p.bX = a->bX; p.bU = nU ? a->bU : nullptr; p.Kc = nU ? a->Kc : nullptr;
    const long long per = (p.K + 1LL) * p.nX + (long long)p.K * nU * (1LL + p.nX);
    const int block = 256;
    long long gx = (per + 4LL * block - 1) / (4LL * block);   // about four elements per lane
    if (gx > 4096) gx = 4096;
    long long gy = p.G * p.M;
    if (gy > 65535) gy = 65535;                               // the kernel strides over the rest
    candidates_kernel<<<dim3((unsigned)gx, (unsigned)gy), block, 0, (cudaStream_t)stream>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    return TREPB_OK;
}

extern "C" int trepb_candidates_batch(int device, const trepb_candidates_args* a) {
    TREPB_NVTX("trepb_candidates_batch");
    const int c = candidates_check(a);
    if (c >= 0) return c;
    const size_t G = (size_t)a->groups, M = (size_t)a->ncand, K = (size_t)a->nsteps, nX = (size_t)a->nX, nU = (size_t)a->nU;
    // the rollouts the groups read: rows[] indexes nrollouts of them (without rows, one per group)
    const size_t Rn = a->rows ? (size_t)a->nrollouts : G, d = 8;
    const void* const src[7] = {a->rows, a->lam, a->X, a->U, a->dX, a->dU, a->Kproj};
    const size_t in_b[7] = {G * 4, M * d, Rn * (K + 1) * nX * d, Rn * K * nU * d, Rn * (K + 1) * nX * d, Rn * K * nU * d,
                            Rn * K * nU * nX * d};
    void* const dst[3] = {a->bX, a->bU, a->Kc};
    const size_t out_b[3] = {G * M * (K + 1) * nX * d, G * M * K * nU * d, G * M * K * nU * nX * d};
    return stage_bytes(device, src, in_b, dst, out_b, [&](void* const* i, void* const* o) {
        trepb_candidates_args x = *a;
        x.rows = (const int32_t*)i[0]; x.lam = (const double*)i[1]; x.X = (const double*)i[2]; x.U = (const double*)i[3];
        x.dX = (const double*)i[4]; x.dU = (const double*)i[5]; x.Kproj = (const double*)i[6];
        x.bX = (double*)o[0]; x.bU = (double*)o[1]; x.Kc = (double*)o[2];
        return trepb_candidates_batch_dev(device, &x, nullptr);
    });
}

// ---- stationary LQR: the discrete algebraic Riccati equation (trepb_dare.cuh) -------------------------------------
namespace {
static_assert(TREPB_DARE_SINGULAR == ST_SINGULAR, "a singular DARE solve reports the LQR kernel's code");

// the checks both DARE entry points make before any CUDA call; -1 = go on
int dare_check(const trepb_dare_args* a) {
    if (!a) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    if (a->batch < 0 || a->nX < 1 || a->nU < 1 || a->max_iterations < 1) return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    if (!(a->tol > 0.0)) return lqr_fail(TREPB_ERR_INVALID, "tol must be positive");
    const void* req[5] = {a->A, a->B, a->Q, a->R, a->status};
    const char* names[5] = {"A", "B", "Q", "R", "status"};
    std::string miss;
    for (int i = 0; i < 5; ++i)
        if (!req[i]) miss += std::string(miss.empty() ? "" : ", ") + names[i];
    if (!miss.empty()) return lqr_fail(TREPB_ERR_INVALID, "A, B, Q, R and status are required (missing: " + miss + ")");
    if (a->batch == 0) return TREPB_OK;
    return -1;
}

int dare_launch(int device, const DareParams& p, cudaStream_t stream) {
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    const DareLayout L = dare_layout(p.nX, p.nU);
    const size_t smem = (size_t)L.total * sizeof(double);
    int smem_optin = 0, sms = 0;
    e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    if (smem > (size_t)smem_optin)
        return lqr_fail(TREPB_ERR_UNSUPPORTED, "state / input dimensions too large for the shared-memory DARE solve");
    e = cudaFuncSetAttribute((const void*)dare_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    const int block = 32 * L.nw;
    // small models: as many CTAs per SM as shared memory allows (one model per CTA at a time)
    int occ = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dare_kernel, block, smem) != cudaSuccess || occ < 1) occ = 1;
    const long long slots = (long long)sms * occ;
    const long long grid = p.batch < slots ? p.batch : slots;
    dare_kernel<<<(int)grid, block, smem, stream>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    return TREPB_OK;
}
}  // namespace

extern "C" int trepb_dare_batch_dev(int device, const trepb_dare_args* a, void* stream) {
    TREPB_NVTX("trepb_dare_batch_dev");
    const int c = dare_check(a);
    if (c >= 0) return c;
    const long long nX = a->nX, nU = a->nU;
    DareParams p{};
    p.batch = a->batch; p.nX = a->nX; p.nU = a->nU; p.max_it = a->max_iterations; p.tol = a->tol;
    p.A = a->A; p.B = a->B; p.Q = a->Q; p.R = a->R; p.S = a->S;
    p.Qs = a->q_per_rollout ? nX * nX : 0; p.Rs = a->r_per_rollout ? nU * nU : 0; p.Ss = a->s_per_rollout ? nX * nU : 0;
    p.K = a->K; p.P = a->P; p.status = a->status; p.iters = a->iterations;
    return dare_launch(device, p, (cudaStream_t)stream);
}

extern "C" int trepb_dare_batch(int device, const trepb_dare_args* a) {
    TREPB_NVTX("trepb_dare_batch");
    const int c = dare_check(a);
    if (c >= 0) return c;
    const size_t Rn = (size_t)a->batch, nX = (size_t)a->nX, nU = (size_t)a->nU, d = 8;
    const void* const src[5] = {a->A, a->B, a->Q, a->R, a->S};
    const size_t in_b[5] = {Rn * nX * nX * d, Rn * nX * nU * d, (a->q_per_rollout ? Rn : 1) * nX * nX * d,
                            (a->r_per_rollout ? Rn : 1) * nU * nU * d, (a->s_per_rollout ? Rn : 1) * nX * nU * d};
    void* const dst[4] = {a->K, a->P, a->status, a->iterations};
    const size_t out_b[4] = {Rn * nU * nX * d, Rn * nX * nX * d, Rn * 4, Rn * 4};
    return stage_bytes(device, src, in_b, dst, out_b, [&](void* const* i, void* const* o) {
        trepb_dare_args x = *a;
        x.A = (const double*)i[0]; x.B = (const double*)i[1]; x.Q = (const double*)i[2]; x.R = (const double*)i[3];
        x.S = (const double*)i[4];
        x.K = (double*)o[0]; x.P = (double*)o[1]; x.status = (int32_t*)o[2]; x.iterations = (int32_t*)o[3];
        return trepb_dare_batch_dev(device, &x, nullptr);
    });
}

// ---- closed-loop cost and stability of stationary gains: the discrete Lyapunov equation (trepb_dlyap.cuh) --------
namespace {
// the checks both Lyapunov entry points make before any CUDA call; -1 = go on
int dlyap_check(const trepb_dlyap_args* a) {
    if (!a) return lqr_fail(TREPB_ERR_INVALID, "null argument");
    if (a->pairs < 0 || a->gains < 0 || a->models < 0 || a->nX < 1 || a->nU < 1 || a->max_iterations < 1)
        return lqr_fail(TREPB_ERR_INVALID, "bad sizes");
    if (!(a->tol > 0.0)) return lqr_fail(TREPB_ERR_INVALID, "tol must be positive");
    const void* req[6] = {a->A, a->B, a->K, a->Q, a->R, a->status};
    const char* names[6] = {"A", "B", "K", "Q", "R", "status"};
    std::string miss;
    for (int i = 0; i < 6; ++i)
        if (!req[i]) miss += std::string(miss.empty() ? "" : ", ") + names[i];
    if (!miss.empty()) return lqr_fail(TREPB_ERR_INVALID, "A, B, K, Q, R and status are required (missing: " + miss + ")");
    if (a->x0 && a->W) return lqr_fail(TREPB_ERR_INVALID, "x0 and W are exclusive");
    if (a->cost && !a->x0 && !a->W) return lqr_fail(TREPB_ERR_INVALID, "cost needs x0 or W");
    if (a->pairs == 0) return TREPB_OK;
    if (!a->gain_index && a->gains < a->pairs)
        return lqr_fail(TREPB_ERR_INVALID, "without gain_index pair p evaluates gain p: gains must be >= pairs");
    if (!a->model_index && a->models < a->pairs)
        return lqr_fail(TREPB_ERR_INVALID, "without model_index pair p runs under model p: models must be >= pairs");
    return -1;
}

// the host form's index check (the _dev form's kernel reports TREPB_DLYAP_BAD_INDEX instead)
int dlyap_check_index(const int32_t* idx, long long pairs, long long count, const char* name) {
    if (!idx) return -1;
    for (long long p = 0; p < pairs; ++p)
        if (idx[p] < 0 || idx[p] >= count)
            return lqr_fail(TREPB_ERR_INVALID, std::string(name) + "[" + std::to_string(p) + "] = " +
                                                   std::to_string(idx[p]) + " is outside [0, " + std::to_string(count) + ")");
    return -1;
}

int dlyap_launch(int device, const DlyapParams& p, cudaStream_t stream) {
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    const DlyapLayout L = dlyap_layout(p.nX, p.nU);
    const size_t smem = (size_t)L.total * sizeof(double);
    int smem_optin = 0, sms = 0;
    e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    if (smem > (size_t)smem_optin)
        return lqr_fail(TREPB_ERR_UNSUPPORTED, "state / input dimensions too large for the shared-memory Lyapunov solve: " +
                                                   std::to_string(smem) + " bytes of shared memory needed, " +
                                                   std::to_string(smem_optin) + " per block on this device");
    e = cudaFuncSetAttribute((const void*)dlyap_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    const int block = 32 * L.nw;
    // small states: as many CTAs per SM as shared memory allows (one pair per CTA at a time)
    int occ = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, dlyap_kernel, block, smem) != cudaSuccess || occ < 1) occ = 1;
    const long long slots = (long long)sms * occ;
    const long long grid = p.pairs < slots ? p.pairs : slots;
    dlyap_kernel<<<(int)grid, block, smem, stream>>>(p);
    e = cudaGetLastError();
    if (e != cudaSuccess) return lqr_fail(TREPB_ERR_CUDA, cudaGetErrorString(e));
    return TREPB_OK;
}
}  // namespace

extern "C" int trepb_dlyap_batch_dev(int device, const trepb_dlyap_args* a, void* stream) {
    TREPB_NVTX("trepb_dlyap_batch_dev");
    const int c = dlyap_check(a);
    if (c >= 0) return c;
    const long long nX = a->nX, nU = a->nU;
    DlyapParams p{};
    p.pairs = a->pairs; p.G = a->gains; p.M = a->models;
    p.nX = a->nX; p.nU = a->nU; p.max_it = a->max_iterations; p.tol = a->tol;
    p.A = a->A; p.B = a->B; p.K = a->K; p.Q = a->Q; p.R = a->R; p.S = a->S;
    p.Qs = a->q_per_model ? nX * nX : 0; p.Rs = a->r_per_model ? nU * nU : 0; p.Ss = a->s_per_model ? nX * nU : 0;
    p.gidx = a->gain_index; p.midx = a->model_index;
    p.x0 = a->cost ? a->x0 : nullptr; p.W = a->cost ? a->W : nullptr; p.xs = a->x0_per_pair ? nX : 0;
    p.P = a->P; p.cost = a->cost; p.status = a->status; p.iters = a->iterations;
    return dlyap_launch(device, p, (cudaStream_t)stream);
}

extern "C" int trepb_dlyap_batch(int device, const trepb_dlyap_args* a) {
    TREPB_NVTX("trepb_dlyap_batch");
    int c = dlyap_check(a);
    if (c >= 0) return c;
    if ((c = dlyap_check_index(a->gain_index, a->pairs, a->gains, "gain_index")) >= 0) return c;
    if ((c = dlyap_check_index(a->model_index, a->pairs, a->models, "model_index")) >= 0) return c;
    const size_t Pn = (size_t)a->pairs, d = 8, nX = (size_t)a->nX, nU = (size_t)a->nU;
    // the arrays cover the gains / models the indices reach (without an index: the first `pairs`)
    const size_t G = a->gain_index ? (size_t)a->gains : Pn, M = a->model_index ? (size_t)a->models : Pn;
    const void* const src[10] = {a->A, a->B, a->K, a->Q, a->R, a->S, a->gain_index, a->model_index,
                                 a->cost ? a->x0 : nullptr, a->cost ? a->W : nullptr};
    const size_t in_b[10] = {M * nX * nX * d, M * nX * nU * d, G * nU * nX * d, (a->q_per_model ? M : 1) * nX * nX * d,
                             (a->r_per_model ? M : 1) * nU * nU * d, (a->s_per_model ? M : 1) * nX * nU * d, Pn * 4,
                             Pn * 4, (a->x0_per_pair ? Pn : 1) * nX * d, nX * nX * d};
    void* const dst[4] = {a->P, a->cost, a->status, a->iterations};
    const size_t out_b[4] = {Pn * nX * nX * d, Pn * d, Pn * 4, Pn * 4};
    return stage_bytes(device, src, in_b, dst, out_b, [&](void* const* i, void* const* o) {
        trepb_dlyap_args x = *a;
        x.A = (const double*)i[0]; x.B = (const double*)i[1]; x.K = (const double*)i[2]; x.Q = (const double*)i[3];
        x.R = (const double*)i[4]; x.S = (const double*)i[5];
        x.gain_index = (const int32_t*)i[6]; x.model_index = (const int32_t*)i[7];
        x.x0 = (const double*)i[8]; x.W = (const double*)i[9];
        x.P = (double*)o[0]; x.cost = (double*)o[1]; x.status = (int32_t*)o[2]; x.iterations = (int32_t*)o[3];
        x.gains = (int64_t)G; x.models = (int64_t)M;
        return trepb_dlyap_batch_dev(device, &x, nullptr);
    });
}
