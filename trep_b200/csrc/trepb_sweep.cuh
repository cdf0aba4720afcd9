// Tangent (forward) and adjoint (backward) sweeps over a linearization that is already in HBM: the two linear
// recursions of a descent direction that remain once linearize, the Riccati sweep and the LQ solve have run.
//
//   tangent  (DSystem.dproject, trep/discopt/dsystem.py:460-471; the end of DOptimizer.calc_descent_direction,
//             doptimizer.py:348-402):
//       dX[0] = x0 (default bdX[0]);  dU[k] = bdU[k] - K[k] (dX[k] - bdX[k]);  dX[k+1] = A[k] dX[k] + B[k] dU[k]
//   adjoint  (the costate of DOptimizer.calc_newton_model, doptimizer.py:319-345):
//       z[K] = m_dx;  z[k] = l_dx[k] + A[k]^T z[k+1] - K[k]^T (l_du[k] + B[k]^T z[k+1])
//       (K NULL: the open-loop costate z[k] = l_dx[k] + A[k]^T z[k+1])
//
// A, B, K are read in the layouts trepb_linearize_batch_dev ([rollout][k], rollout-major instances) and
// trepb_lqr_batch_dev / trepb_lq_batch_dev write, so no copy or transpose sits between the calls.  The work is
// sequential in k and independent over rollouts: a team of `team` lanes (a power of two >= max(nX, nU)) owns one
// rollout, several teams share a CTA for small states.  Step k's A / B / K and its two vectors are staged in
// shared memory by cp.async `stages - 1` steps ahead (coalesced 8-byte copies: the rows are padded to an odd
// length, so the tangent sweep's row-per-lane reads of A, B and K are free of bank conflicts, and the adjoint
// sweep reads columns, which are contiguous across lanes anyway).  Every output element is summed by one lane in a
// fixed order (j ascending), so a rollout's bits do not depend on the batch, the grid or its team's placement.
#pragma once
#include <cuda_runtime.h>

namespace trepb {
namespace {

struct SweepParams {
    long long batch;
    int K, nX, nU;
    const double *A, *B, *Kfb;    // [batch][K][nX][nX], [batch][K][nX][nU], [batch][K][nU][nX] (Kfb may be null)
    const double *vx, *vu;        // tangent: bdX [batch][K+1][nX], bdU [batch][K][nU]; adjoint: l_dx [batch][K][nX],
                                  // l_du [batch][K][nU]; null = zero
    const double* x0;             // tangent: dX[0] [batch][nX] (null: bdX[0], or zero); adjoint: m_dx [batch][nX]
    double *ox, *ou;              // tangent: dX [batch][K+1][nX], dU [batch][K][nU];
                                  // adjoint: z [batch][K+1][nX], z1 [batch][K][nX] = z[k+1] (may be null)
    int team, stages;             // lanes per rollout (teams per CTA = blockDim.x / team), cp.async ring depth
};

// padded row lengths and the doubles of one staged step: A [nX][ldx], B [nX][ldu], K [nU][ldx], vx [nX], vu [nU]
__host__ __device__ __forceinline__ int sweep_ldx(int nX) { return nX | 1; }
__host__ __device__ __forceinline__ int sweep_ldu(int nU) { return nU | 1; }
__host__ __device__ __forceinline__ long long sweep_stage(int nX, int nU) {
    const long long s = (long long)nX * sweep_ldx(nX) + (long long)nX * sweep_ldu(nU) + (long long)nU * sweep_ldx(nX) + nX + nU;
    return (s + 1) & ~1LL;
}
// per team: the stage ring, then two state vectors (ping-pong) and one input-sized vector
__host__ __device__ __forceinline__ long long sweep_team_doubles(int nX, int nU, int stages) {
    return stages * sweep_stage(nX, nU) + 2LL * nX + nU + 2;
}

// rows x cols doubles from src (dense rows) to dst (rows of length ld), lanes t, t + T, ... of a team
__device__ __forceinline__ void sweep_copy(double* dst, int ld, const double* src, int rows, int cols, int t, int T) {
    if (rows <= 0 || cols <= 0) return;
    const unsigned d0 = (unsigned)__cvta_generic_to_shared(dst);
    const int di = T / cols, dj = T - di * cols;   // (row, column) step of element e -> e + T
    int i = t / cols, j = t - i * cols;
    for (int e = t; e < rows * cols; e += T) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d0 + 8u * (unsigned)(i * ld + j)), "l"(src + e) : "memory");
        i += di; j += dj;
        if (j >= cols) { j -= cols; ++i; }
    }
}
__device__ __forceinline__ void sweep_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// wait until at most `pending` (= stages - 2) groups of this thread are still in flight
__device__ __forceinline__ void sweep_wait(int pending) {
    switch (pending) {
        case 6: asm volatile("cp.async.wait_group 6;" ::: "memory"); break;
        case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
        default: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    }
}

// step `k` of rollout r into the stage at S (tangent: vx = bdX[k]; adjoint: vx = l_dx[k])
__device__ __forceinline__ void sweep_issue(const SweepParams& p, double* S, long long r, int k, int t, int T, bool tangent) {
    const int nX = p.nX, nU = p.nU, ldx = sweep_ldx(nX), ldu = sweep_ldu(nU);
    const long long rk = r * p.K + k;
    double* As = S;
    double* Bs = As + nX * ldx;
    double* Ks = Bs + nX * ldu;
    double* vx = Ks + nU * ldx;
    double* vu = vx + nX;
    sweep_copy(As, ldx, p.A + rk * nX * nX, nX, nX, t, T);
    if (nU) {
        if (p.B) sweep_copy(Bs, ldu, p.B + rk * nX * nU, nX, nU, t, T);
        if (p.Kfb) sweep_copy(Ks, ldx, p.Kfb + rk * nU * nX, nU, nX, t, T);
        if (p.vu) sweep_copy(vu, nU, p.vu + rk * nU, 1, nU, t, T);
    }
    if (p.vx) sweep_copy(vx, nX, p.vx + (tangent ? r * (p.K + 1LL) + k : rk) * nX, 1, nX, t, T);
}

template <bool TANGENT>
__global__ void __launch_bounds__(128) sweep_kernel(const SweepParams p) {
    extern __shared__ __align__(16) double sm[];
    const int nX = p.nX, nU = p.nU, K = p.K, T = p.team, S = p.stages;
    const int ldx = sweep_ldx(nX), ldu = sweep_ldu(nU);
    const long long st = sweep_stage(nX, nU);
    const int G = blockDim.x / T, g = threadIdx.x / T, t = threadIdx.x - g * T;
    double* ring = sm + g * sweep_team_doubles(nX, nU, S);
    double* const xa = ring + S * st;                       // dX[k] / z[k+1] and the next one (ping-pong)
    double* const xb = xa + nX;
    double* const uv = xb + nX;                             // dU[k] / g = l_du[k] + B[k]^T z[k+1]
    const bool use_k = p.Kfb != nullptr && nU > 0;
    for (long long base = (long long)blockIdx.x * G; base < p.batch; base += (long long)gridDim.x * G) {
        const long long r = base + g;
        const bool active = r < p.batch;
        // prologue: the first stages - 1 steps in flight (empty groups keep every thread's count the same)
        for (int s = 0; s < S - 1; ++s) {
            if (active && s < K) sweep_issue(p, ring + s * st, r, TANGENT ? s : K - 1 - s, t, T, TANGENT);
            sweep_commit();
        }
        if (active) {
            double* x = xa;
            if (TANGENT) {
                const double* src = p.x0 ? p.x0 + r * nX : p.vx ? p.vx + r * (K + 1LL) * nX : nullptr;
                for (int i = t; i < nX; i += T) {
                    const double v = src ? src[i] : 0.0;
                    x[i] = v;
                    p.ox[r * (K + 1LL) * nX + i] = v;
                }
            } else {
                for (int i = t; i < nX; i += T) {
                    const double v = p.x0[r * nX + i];
                    x[i] = v;
                    p.ox[(r * (K + 1LL) + K) * nX + i] = v;
                    if (p.ou) p.ou[(r * K + K - 1) * nX + i] = v;
                }
            }
        }
        for (int it = 0; it < K; ++it) {
            const int k = TANGENT ? it : K - 1 - it;
            sweep_wait(S - 2);                                  // step k has landed (this thread's copies)
            __syncthreads();                                    // ... and every other lane's
            {   // the slot of step it - 1 is free: fetch step it + S - 1 into it
                const int nxt = it + S - 1;
                if (active && nxt < K) sweep_issue(p, ring + (nxt % S) * st, r, TANGENT ? nxt : K - 1 - nxt, t, T, TANGENT);
                sweep_commit();
            }
            const double* As = ring + (it % S) * st;
            const double* Bs = As + nX * ldx;
            const double* Ks = Bs + nX * ldu;
            const double* vx = Ks + nU * ldx;
            const double* vu = vx + nX;
            const double* x = (it & 1) ? xb : xa;
            double* xn = (it & 1) ? xa : xb;
            if (TANGENT) {
                // dU[k] = bdU[k] - K[k] (dX[k] - bdX[k])
                if (active)
                    for (int i = t; i < nU; i += T) {
                        double acc = p.vu ? vu[i] : 0.0;
                        const double* Ki = Ks + i * ldx;
                        if (p.vx) for (int j = 0; j < nX; ++j) acc -= Ki[j] * (x[j] - vx[j]);
                        else for (int j = 0; j < nX; ++j) acc -= Ki[j] * x[j];
                        uv[i] = acc;
                        p.ou[(r * K + k) * nU + i] = acc;
                    }
                __syncthreads();
                // dX[k+1] = A[k] dX[k] + B[k] dU[k]
                if (active)
                    for (int i = t; i < nX; i += T) {
                        double acc = 0.0;
                        const double* Ai = As + i * ldx;
                        for (int j = 0; j < nX; ++j) acc += Ai[j] * x[j];
                        const double* Bi = Bs + i * ldu;
                        for (int j = 0; j < nU; ++j) acc += Bi[j] * uv[j];
                        xn[i] = acc;
                        p.ox[(r * (K + 1LL) + k + 1) * nX + i] = acc;
                    }
            } else {
                // g = l_du[k] + B[k]^T z[k+1], once per step
                if (use_k) {
                    if (active)
                        for (int i = t; i < nU; i += T) {
                            double acc = p.vu ? vu[i] : 0.0;
                            for (int j = 0; j < nX; ++j) acc += Bs[j * ldu + i] * x[j];
                            uv[i] = acc;
                        }
                    __syncthreads();
                }
                // z[k] = l_dx[k] + A[k]^T z[k+1] - K[k]^T g
                if (active)
                    for (int i = t; i < nX; i += T) {
                        double acc = p.vx ? vx[i] : 0.0;
                        for (int j = 0; j < nX; ++j) acc += As[j * ldx + i] * x[j];
                        if (use_k) for (int j = 0; j < nU; ++j) acc -= Ks[j * ldx + i] * uv[j];
                        xn[i] = acc;
                        p.ox[(r * (K + 1LL) + k) * nX + i] = acc;
                        if (p.ou && k > 0) p.ou[(r * K + k - 1) * nX + i] = acc;
                    }
            }
        }
        sweep_wait(0);
        __syncthreads();                                        // the ring is reused by the next rollout group
    }
}

}  // namespace
}  // namespace trepb
