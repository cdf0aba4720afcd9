// The quadratic tracking cost of trep.discopt.DCost (dcost.py) as DOptimizer sums it (doptimizer.py calc_cost /
// calc_dcost), its LQ model, and the Armijo line-search candidates, batched over trajectories.
//
//   dx_k = X[k] - Xd[k],  du_k = U[k] - Ud[k]   (trajectory b tracks reference ref[b], or 0)
//   cost  = sum_{k<K} (dx_k^T Q dx_k + du_k^T R du_k) / 2 + dx_K^T Q dx_K / 2
//   q[k]  = dx_k^T Q (k = 0..K),  r[k] = du_k^T R
//   dcost = sum_{k<K} (q[k] . dX[k] + r[k] . dU[k]) + q[K] . dX[K]
//   model Qm[k] = Q (+ fdxdx[k], k < K),  Sm[k] = 0 (+ fdxdu[k]),  Rm[k] = R (+ fdudu[k])
//
// track_kernel runs two kinds of CTA in one launch.  The first `cost_blocks` CTAs each own whole trajectories
// (the cost and gradient role): a tile of steps is staged in shared memory as [dx | du], one lane per (step,
// column) forms q / r, one lane per step forms its cost and dcost terms, and lane 0 adds the per-step terms in
// ascending k.  Every sum (over i, j and k) is a chain of separately rounded products and additions in ascending
// index order, so its bits depend on neither the batch, the tile length nor the grid.  The other CTAs stream the
// model slabs (the memory-bound part: Q + fdxdx alone is nX^2 doubles read and written per step) with one IEEE
// addition per element, so Qm equals the host's Q + fdxdx bit for bit.
//
// candidates_kernel writes bX[g][m] = X + lam[m] dX, bU[g][m] = U + lam[m] dU (product and sum rounded
// separately, as numpy's X + lam * dX) and one copy of the gains per candidate, for rollout rows[g].
#pragma once
#include <cuda_runtime.h>

namespace trepb {
namespace {

struct TrackParams {
    long long batch;
    int K, nX, nU;
    const double *X, *U, *Xd, *Ud, *Q, *R;   // [batch][K+1][nX], [batch][K][nU], [nref][K+1][nX], [nref][K][nU]
    const int* ref;                          // [batch] reference of each trajectory, null = 0
    const double *dX, *dU;                   // [batch][K+1][nX], [batch][K][nU] (dcost)
    const double *fxx, *fxu, *fuu;           // [batch*K][nX][nX], [batch*K][nX][nU], [batch*K][nU][nU], null = none
    double *cost, *dcost, *q, *r, *l_dx, *m_dx;
    double *Qm, *Sm, *Rm;                    // [batch][K+1][nX][nX], [batch][K][nX][nU], [batch][K][nU][nU]
    int cost_blocks, tile, model_bpt;        // CTAs of the cost role, steps per staged tile, model CTAs per trajectory
};

// doubles of shared memory a cost-role CTA needs for a tile of `tile` steps: [dx|du] and [q|r], then two scalars
__host__ __device__ __forceinline__ long long track_smem_doubles(int nX, int nU, int tile) {
    return 2LL * tile * (nX + nU) + 2LL * tile;
}

__device__ __forceinline__ void track_cost_role(const TrackParams& p, double* sm, long long b) {
    const int nX = p.nX, nU = p.nU, K = p.K, C = nX + nU, TK = p.tile, T = blockDim.x, t = threadIdx.x;
    double* dv = sm;                      // [TK][C] dx | du
    double* gv = dv + (long long)TK * C;  // [TK][C] q  | r
    double* ck = gv + (long long)TK * C;  // [TK] cost term of each step
    double* dk = ck + TK;                 // [TK] dcost term of each step
    const long long rf = p.ref ? p.ref[b] : 0;
    const double* X = p.X + b * (K + 1LL) * nX;
    const double* U = nU ? p.U + b * (long long)K * nU : nullptr;
    const double* Xd = p.Xd + rf * (K + 1LL) * nX;
    const double* Ud = nU ? p.Ud + rf * (long long)K * nU : nullptr;
    const bool want_d = p.dcost != nullptr;
    double cost = 0.0, dcost = 0.0;       // lane 0's running sums over k
    for (int k0 = 0; k0 <= K; k0 += TK) {
        const int nk = (K + 1 - k0) < TK ? (K + 1 - k0) : TK;
        for (int e = t; e < nk * C; e += T) {
            const int kl = e / C, j = e - kl * C, k = k0 + kl;
            double v = 0.0;
            if (j < nX) v = __dsub_rn(X[(long long)k * nX + j], Xd[(long long)k * nX + j]);
            else if (k < K) v = __dsub_rn(U[(long long)k * nU + j - nX], Ud[(long long)k * nU + j - nX]);
            dv[e] = v;
        }
        __syncthreads();
        // q[k][j] = sum_i dx_i Q[i][j],  r[k][j] = sum_i du_i R[i][j]  (ascending i, one lane per (k, j))
        for (int e = t; e < nk * C; e += T) {
            const int kl = e / C, j = e - kl * C, k = k0 + kl;
            const double* d = dv + kl * C;
            double acc = 0.0;
            if (j < nX) {
                for (int i = 0; i < nX; ++i) acc = __dadd_rn(acc, __dmul_rn(d[i], p.Q[i * nX + j]));
                const long long o = (b * (K + 1LL) + k) * nX + j;
                if (p.q) p.q[o] = acc;
                if (k < K) { if (p.l_dx) p.l_dx[(b * K + k) * nX + j] = acc; }
                else if (p.m_dx) p.m_dx[b * nX + j] = acc;
            } else if (k < K) {
                const int ju = j - nX;
                for (int i = 0; i < nU; ++i) acc = __dadd_rn(acc, __dmul_rn(d[nX + i], p.R[i * nU + ju]));
                if (p.r) p.r[(b * K + k) * nU + ju] = acc;
            }
            gv[e] = acc;
        }
        __syncthreads();
        // the step's terms: (dx.q + du.r) / 2 and q.dX + r.dU, ascending j
        for (int kl = t; kl < nk; kl += T) {
            const int k = k0 + kl;
            const double* d = dv + kl * C;
            const double* g = gv + kl * C;
            double xq = 0.0, ur = 0.0;
            for (int j = 0; j < nX; ++j) xq = __dadd_rn(xq, __dmul_rn(d[j], g[j]));
            if (k < K) for (int j = nX; j < C; ++j) ur = __dadd_rn(ur, __dmul_rn(d[j], g[j]));
            ck[kl] = __dmul_rn(0.5, k < K ? __dadd_rn(xq, ur) : xq);
            if (want_d) {
                const double* dX = p.dX + (b * (K + 1LL) + k) * nX;
                double sx = 0.0, su = 0.0;
                for (int j = 0; j < nX; ++j) sx = __dadd_rn(sx, __dmul_rn(g[j], dX[j]));
                if (k < K) {
                    const double* dU = p.dU + (b * K + k) * nU;
                    for (int j = 0; j < nU; ++j) su = __dadd_rn(su, __dmul_rn(g[nX + j], dU[j]));
                }
                dk[kl] = k < K ? __dadd_rn(sx, su) : sx;
            }
        }
        __syncthreads();
        if (t == 0)
            for (int kl = 0; kl < nk; ++kl) {
                cost = __dadd_rn(cost, ck[kl]);
                if (want_d) dcost = __dadd_rn(dcost, dk[kl]);
            }
        __syncthreads();                  // the tile's buffers are refilled next
    }
    if (t == 0) {
        if (p.cost) p.cost[b] = cost;
        if (want_d) p.dcost[b] = dcost;
    }
}

__device__ __forceinline__ void track_model_role(const TrackParams& p, long long w, long long nw) {
    const int nX = p.nX, nU = p.nU, K = p.K, T = blockDim.x;
    const unsigned xx = (unsigned)nX * nX, xu = (unsigned)nX * nU, uu = (unsigned)nU * nU;
    const unsigned segQ = (unsigned)(K + 1) * xx, segS = p.Sm ? (unsigned)K * xu : 0u, segR = p.Rm ? (unsigned)K * uu : 0u;
    const unsigned per = segQ + segS + segR;
    const long long bpt = p.model_bpt;
    for (; w < p.batch * bpt; w += nw) {
        const long long b = w / bpt;
        const unsigned lb = (unsigned)(w - b * bpt);
        for (unsigned e = lb * T + threadIdx.x; e < per; e += (unsigned)bpt * T) {
            if (e < segQ) {
                const unsigned k = e / xx, ij = e - k * xx;
                double v = p.Q[ij];
                if (p.fxx && (int)k < K) v = __dadd_rn(v, p.fxx[(b * K + k) * xx + ij]);
                p.Qm[b * segQ + e] = v;
            } else if (e < segQ + segS) {
                const unsigned f = e - segQ;
                p.Sm[b * (long long)K * xu + f] = p.fxu ? p.fxu[b * (long long)K * xu + f] : 0.0;
            } else {
                const unsigned f = e - segQ - segS, k = f / uu, ij = f - k * uu;
                double v = p.R[ij];
                if (p.fuu) v = __dadd_rn(v, p.fuu[(b * K + k) * uu + ij]);
                p.Rm[b * (long long)K * uu + f] = v;
            }
        }
    }
}

__global__ void __launch_bounds__(256) track_kernel(const TrackParams p) {
    extern __shared__ __align__(16) double tsm[];
    if ((int)blockIdx.x < p.cost_blocks) {
        for (long long b = blockIdx.x; b < p.batch; b += p.cost_blocks) track_cost_role(p, tsm, b);
    } else {
        track_model_role(p, (long long)blockIdx.x - p.cost_blocks, (long long)gridDim.x - p.cost_blocks);
    }
}

struct CandParams {
    long long G;
    int M, K, nX, nU;
    const int* rows;                          // [G] rollout of group g, null = g
    const double* lam;                        // [M]
    const double *X, *U, *dX, *dU, *Kp;       // [R][K+1][nX], [R][K][nU], same, same, [R][K][nU][nX]
    double *bX, *bU, *Kc;                     // [G][M][K+1][nX], [G][M][K][nU], [G][M][K][nU][nX]
};

__global__ void __launch_bounds__(256) candidates_kernel(const CandParams p) {
    const unsigned sx = (unsigned)(p.K + 1) * p.nX, su = (unsigned)p.K * p.nU, sk = su * p.nX;
    const unsigned per = sx + su + sk;
    for (long long c = blockIdx.y; c < p.G * p.M; c += gridDim.y) {
        const long long g = c / p.M;
        const int m = (int)(c - g * p.M);
        const long long r = p.rows ? p.rows[g] : g;
        const double lam = p.lam[m];
        for (unsigned e = blockIdx.x * blockDim.x + threadIdx.x; e < per; e += gridDim.x * blockDim.x) {
            if (e < sx) {
                p.bX[c * sx + e] = __dadd_rn(p.X[r * sx + e], __dmul_rn(lam, p.dX[r * sx + e]));
            } else if (e < sx + su) {
                const unsigned f = e - sx;
                p.bU[c * su + f] = __dadd_rn(p.U[r * su + f], __dmul_rn(lam, p.dU[r * su + f]));
            } else {
                const unsigned f = e - sx - su;
                p.Kc[c * sk + f] = p.Kp[r * sk + f];
            }
        }
    }
}

}  // namespace
}  // namespace trepb
