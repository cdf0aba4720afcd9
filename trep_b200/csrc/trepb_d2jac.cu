// Kernels of the O(nx) second-derivative path (trepb_d2jac.cuh): directional derivative of the
// Jacobian tables on dual numbers (pass A), contraction + solves per parameter pair (pass B).
#include "trepb_d2jac.cuh"

namespace trepb {
// ---------------------------------------------------------------------------------------------
// pass A kernel
// ---------------------------------------------------------------------------------------------
// Each thread owns one (instance, s) record of jl.size doubles; the 32 records of a warp are
// consecutive in G.  Values are staged through a 32 x 32 shared-memory tile per warp so that every
// store instruction writes 256 contiguous bytes of one record.
struct TileSink {
    double* tile;        // [32][33] of this warp
    double* G0;          // record of lane 0
    int size, rows, lane, k;
    long e0;
    __device__ __forceinline__ void push(double v) {
        tile[lane * 33 + k] = v;
        if (++k == 32) flush();
    }
    __device__ __forceinline__ void flush() {
        __syncwarp();
        if (lane < k) {
            for (int r = 0; r < rows; ++r) G0[(long)r * size + e0 + lane] = tile[r * 33 + lane];
        }
        e0 += k;
        k = 0;
        __syncwarp();
    }
};

#ifndef TREPB_D2JAC_MINB
#define TREPB_D2JAC_MINB 4   // measured on the marionette (B200): 4 CTAs per SM at 128 registers (some spills) 40.8 ms per 4096 instances, 3 at 168: 43.3, 5 at 96: 42.2, 2 at 232: 49.0
#endif
// kVaried: each (instance, s) item expands its instance's parameter row into this thread's slot and points the numeric
// tables of the thread's RtSys copy at it (varied_point).  The integer tables and NzMaps stay in shared memory: NzMaps
// depends on structure only, and an entry that may vary is never a structural zero (varied_check).
template <bool kVaried>
__device__ __forceinline__ void
d2jac_body(const RtSys& rsys, const char* dblob, int blob_bytes, const WsStridedT<Dual>& wsp, const D2Params& p,
           double* __restrict__ G, const JacLayout& jl, long b0, long nb, const VariedArgs& va) {
    extern __shared__ double smem_[];
    const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long nth = (long)gridDim.x * blockDim.x;
    const int n8 = ((blob_bytes + 7) / 8 + 1) & ~1;
    {
        const double* src = (const double*)dblob;
        for (int i = threadIdx.x; i < (blob_bytes + 7) / 8; i += blockDim.x) smem_[i] = src[i];
        __syncthreads();
    }
    std::conditional_t<kVaried, RtSys, const RtSys> sys = rsys.rebased(dblob, (const char*)smem_);
    WsStridedT<Dual> ws = wsp;
    ws.base = wsp.base + tid;
    ws.stride = (unsigned)nth;
    const int lane = threadIdx.x & 31;
    double* tile = smem_ + n8 + (threadIdx.x >> 5) * (32 * 33);
    NzMaps nz;
    nz.place((uint8_t*)(smem_ + n8 + (blockDim.x >> 5) * (32 * 33)), sys.ND(), sys.NK());
    d2jac_build_nz(sys, nz, threadIdx.x, blockDim.x);
    __syncthreads();
    const long total = nb * p.nx;
    for (long g = tid;; g += nth) {
        const long base = g - lane;
        if (base >= total) break;
        const bool in = g < total;
        const long b = b0 + (in ? g / p.nx : 0);
        const int s = in ? (int)(g % p.nx) : 0;
        const bool act = in && !(p.status && p.status[b] != 0);
        if constexpr (kVaried) {
            if (act) varied_point(sys, va.map, va.values + b * va.map.n, va.slots + tid * (long)va.map.n_out);
        }
        if (act) d2jac_eval(sys, ws, nz, p, b, s);
        __syncwarp();
        const double t1 = p.t1 ? p.t1[b] : p.t1s;
        const double t2 = p.t2 ? p.t2[b] : (t1 + p.dts);
        TileSink out;
        out.tile = tile; out.G0 = G + base * jl.size; out.size = jl.size; out.lane = lane; out.k = 0; out.e0 = 0;
        out.rows = total - base < 32 ? (int)(total - base) : 32;
        d2jac_emit(sys, ws, nz, t2 - t1, out);
        if (out.k) out.flush();
    }
}

__global__ void __launch_bounds__(128, TREPB_D2JAC_MINB)
d2jac_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStridedT<Dual> wsp, const D2Params p,
             double* __restrict__ G, const JacLayout jl, long b0, long nb) {
    d2jac_body<false>(rsys, dblob, blob_bytes, wsp, p, G, jl, b0, nb, VariedArgs{});
}
__global__ void __launch_bounds__(128, TREPB_D2JAC_MINB)
d2jac_varied_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStridedT<Dual> wsp, const D2Params p,
                    double* __restrict__ G, const JacLayout jl, long b0, long nb, const VariedArgs va) {
    d2jac_body<true>(rsys, dblob, blob_bytes, wsp, p, G, jl, b0, nb, va);
}

// ---------------------------------------------------------------------------------------------
// pass B kernel: one CTA per (instance, s); thread i works on t = s + i
// shared memory: [Jd nd*nd][Hd nd*nd][JL nc*nd][JC nc*nd][aux al.size][z 2nq][columns (3nd+3nc) x T]
// ---------------------------------------------------------------------------------------------
__global__ void d2solve_kernel(const D2Params p, const double* __restrict__ G, const JacLayout jl, int nd, int nk,
                               int nu, int nc, long b0) {
    extern __shared__ double sm[];
    const int nq = nd + nk, nx = p.nx, T = blockDim.x;
    const long item = blockIdx.x;
    const long bl = item / nx;
    const int s = (int)(item - bl * nx);
    const long b = b0 + bl;
    if (p.status && p.status[b] != 0) return;
    const double* Grow = G + item * jl.size;
    double* Jd = sm;
    double* Hd = Jd + nd * nd;
    double* JL = Hd + nd * nd;
    double* JC = JL + nc * nd;
    double* ax = JC + nc * nd;
    double* zz = ax + p.auxl.size;
    double* cols = zz + 2 * nq;
    for (int i = threadIdx.x; i < nd * nd; i += T) { Jd[i] = Grow[jl.o_q + 4 * i + 1]; Hd[i] = Grow[jl.o_q + 4 * i + 3]; }
    for (int i = threadIdx.x; i < nc * nd; i += T) { JL[i] = Grow[jl.o_jl + i]; JC[i] = Grow[jl.o_jc + i]; }
    const double* aux = p.aux + b * (long)p.auxl.size;
    for (int i = threadIdx.x; i < p.auxl.size; i += T) ax[i] = aux[i];
    if (p.z) for (int i = threadIdx.x; i < 2 * nq; i += T) zz[i] = p.z[b * 2 * nq + i];
    __syncthreads();
    const int t = s + threadIdx.x;
    if (t >= nx) return;
    D2Pair P;
    P.Jd = Jd; P.Hd = Hd; P.JL = JL; P.JC = JC; P.Grow = Grow; P.aux = ax; P.z = p.z ? zz : nullptr;
    P.jl = jl; P.al = p.auxl;
    double* y = cols + threadIdx.x;
    double* lt = y + nd * T;
    double* c = lt + nc * T;
    double* x = c + nd * T;
    double* h = x + nd * T;
    double* hx = h + nc * T;
    d2_pair(P, p, b, nd, nk, nu, nc, s, t, y, lt, c, x, h, hx, T);
}

// ---------------------------------------------------------------------------------------------
// pass B, compile-time sizes (ND dynamic configs, NC constraints): the same arithmetic as d2_pair with
// every per-pair vector in registers and every matrix read as a shared-memory broadcast.
//   * one CTA per instance and PAIR of parameters (sa, sb = nx-1-sa): nx+1 parameter pairs (s, t >= s)
//     per CTA, whatever sa is (one CTA per (instance, s) would leave half the threads without work);
//   * products are accumulated row by row of the matrix (22 independent accumulators per thread,
//     128-bit shared-memory loads), the triangular solves column by column (axpy form: the updates
//     of one column are independent) on transposed LU factors, reciprocal diagonals precomputed;
//   * the only per-thread shared memory is the column used for the pivot gather x[i] = b[piv[i]].
// ---------------------------------------------------------------------------------------------
constexpr int kD2T = 96;   // threads per CTA of the compile-time-size pass B
template <int ND, int NC>
struct D2Ct {
    static constexpr int NCR = NC > 0 ? NC : 1;
    static constexpr int LD = (ND + 1) & ~1;        // row stride of matrices with ND columns
    static constexpr int LP = (NCR + 1) & ~1;       // row stride of matrices with NC columns
    static constexpr int SET = 2 * ND * LD + NC * LD + ND * LP;   // Jd, Hd, JL, JCt
    static constexpr int o_m2t = 2 * SET;
    static constexpr int o_t22 = o_m2t + ND * LD;
    static constexpr int o_dh1 = o_t22 + ND * LD;
    static constexpr int o_dh2t = o_dh1 + NC * LD;
    static constexpr int o_pjt = o_dh2t + ND * LP;
    static constexpr int o_rdm = o_pjt + NCR * LP;
    static constexpr int o_rdp = o_rdm + LD;
    static constexpr int o_piv = o_rdp + LP;                 // ints: pivM[ND], pivP[NC]
    static constexpr int o_z = o_piv + ((ND + NCR + 3) / 4) * 2;
    __host__ __device__ static int o_cols(int nq) { return o_z + ((2 * nq + 1) & ~1); }
    static size_t smem(int nq) { return sizeof(double) * (size_t)(o_cols(nq) + (ND + NCR) * kD2T); }
};

#ifndef TREPB_D2CT_MINB
#define TREPB_D2CT_MINB 3
#endif
template <int ND, int NC>
__global__ void __launch_bounds__(kD2T, TREPB_D2CT_MINB)
d2solve_ct_kernel(const D2Params p, const double* __restrict__ G, const JacLayout jl, int nk, int nu, long b0) {
    using L = D2Ct<ND, NC>;
    constexpr int LD = L::LD, LP = L::LP, NCR = L::NCR, T = kD2T;
    extern __shared__ __align__(16) double sm[];
    const int nq = ND + nk, nx = p.nx;
    const int half = (nx + 1) / 2;
    const long bl = blockIdx.x / half;
    const int sa = (int)(blockIdx.x - bl * half), sb = nx - 1 - sa;
    const long b = b0 + bl;
    if (p.status && p.status[b] != 0) return;
    const int na = nx - sa, tot = na + (sb != sa ? nx - sb : 0);
    const int tid = threadIdx.x;
    // ---- stage the matrices every pair of this CTA shares
    for (int set = 0; set < (sb != sa ? 2 : 1); ++set) {
        const double* Grow = G + (bl * nx + (set ? sb : sa)) * (long)jl.size;
        double* S = sm + set * L::SET;
        for (int e = tid; e < ND * ND; e += T) {
            const int i = e / ND, j = e - i * ND;
            S[i * LD + j] = Grow[jl.o_q + 4 * e + 1];
            S[ND * LD + i * LD + j] = Grow[jl.o_q + 4 * e + 3];
        }
        for (int e = tid; e < NC * ND; e += T) {
            const int c = e / ND, j = e - c * ND;
            S[2 * ND * LD + c * LD + j] = Grow[jl.o_jl + e];
            S[2 * ND * LD + NC * LD + j * LP + c] = Grow[jl.o_jc + e];    // JCt[i][c]
        }
    }
    {
        const double* aux = p.aux + b * (long)p.auxl.size;
        const AuxLayout& al = p.auxl;
        for (int e = tid; e < ND * ND; e += T) {
            const int i = e / ND, j = e - i * ND;
            sm[L::o_m2t + j * LD + i] = aux[al.o_m2 + e];
            sm[L::o_t22 + i * LD + j] = aux[al.o_t22 + e];
        }
        int* piv = (int*)(sm + L::o_piv);
        for (int i = tid; i < ND; i += T) {
            sm[L::o_rdm + i] = 1.0 / aux[al.o_m2 + i * ND + i];
            piv[i] = (int)aux[al.o_m2p + i];
        }
        for (int e = tid; e < NC * ND; e += T) {
            const int c = e / ND, j = e - c * ND;
            sm[L::o_dh1 + c * LD + j] = aux[al.o_dh1 + e];
            sm[L::o_dh2t + j * LP + c] = aux[al.o_dh2 + e];
        }
        for (int e = tid; e < NC * NC; e += T) {
            const int i = e / NC, j = e - i * NC;
            sm[L::o_pjt + j * LP + i] = aux[al.o_pj + e];
        }
        for (int i = tid; i < NC; i += T) {
            sm[L::o_rdp + i] = 1.0 / aux[al.o_pj + i * NC + i];
            piv[ND + i] = (int)aux[al.o_pjp + i];
        }
        if (p.z) for (int i = tid; i < 2 * nq; i += T) sm[L::o_z + i] = p.z[b * 2 * nq + i];
    }
    __syncthreads();
    const double* M2t = sm + L::o_m2t;
    const double* T22 = sm + L::o_t22;
    const double* rdM = sm + L::o_rdm;
    const int* pivM = (const int*)(sm + L::o_piv);
    double* colc = sm + L::o_cols(nq) + tid;
    double* colh = colc + ND * T;
    for (int w = tid; w < tot; w += T) {
        const int set = w < na ? 0 : 1;
        const int s = set ? sb : sa, t = set ? sb + (w - na) : sa + w;
        const double* Grow = G + (bl * nx + s) * (long)jl.size;
        const double* Jd = sm + set * L::SET;
        const double* Hd = Jd + ND * LD;
        const double* JL = Hd + ND * LD;
        const double* JCt = JL + NC * LD;
        int ts, is, tt, it;
        split_param(s, nq, ND, nu, &ts, &is);
        split_param(t, nq, ND, nu, &tt, &it);
        const int cnt_s = ts == 0 ? nq : (ts == 1 ? ND : (ts == 2 ? nu : nk));
        const int cnt_t = tt == 0 ? nq : (tt == 1 ? ND : (tt == 2 ? nu : nk));
        double y[ND], lt[NCR], c[ND], x[ND];
        {
            const double* zt = p.q2_d[tt] + ((long)b * cnt_t + it) * ND;
#pragma unroll
            for (int i = 0; i < ND; ++i) y[i] = zt[i];
            if constexpr (NC > 0) {
                const double* l = p.l1_d[tt] + ((long)b * cnt_t + it) * NC;
#pragma unroll
                for (int cc = 0; cc < NC; ++cc) lt[cc] = l[cc];
            }
        }
        const double* r1 = tt == 0 ? Grow + jl.q(it, 0, ND, 0)
                         : tt == 2 ? Grow + jl.o_ju + it * ND
                         : tt == 3 ? Grow + jl.q(ND + it, 0, ND, 1) : nullptr;
        const double* rh = tt == 0 ? Grow + jl.q(it, 0, ND, 2)
                         : tt == 3 ? Grow + jl.q(ND + it, 0, ND, 3) : nullptr;
        const int r1s = tt == 2 ? 1 : 4;
        // c = -R1 ,  R1 = D^2 F1 [xi_s, xi_t]
#pragma unroll
        for (int j = 0; j < ND; ++j) c[j] = r1 ? r1[j * r1s] : 0.0;
#pragma unroll
        for (int i = 0; i < ND; ++i) {
            const double yi = y[i];
#pragma unroll
            for (int j = 0; j < ND; ++j) c[j] += Jd[i * LD + j] * yi;
        }
        if constexpr (NC > 0) {
#pragma unroll
            for (int cc = 0; cc < NC; ++cc) {
                const double l = lt[cc];
#pragma unroll
                for (int j = 0; j < ND; ++j) c[j] += JL[cc * LD + j] * l;
            }
        }
#pragma unroll
        for (int j = 0; j < ND; ++j) { c[j] = -c[j]; colc[j * T] = c[j]; }
        // x = M2^-1 c
        auto solveM = [&]() {
#pragma unroll
            for (int i = 0; i < ND; ++i) x[i] = colc[pivM[i] * T];
#pragma unroll
            for (int j = 0; j < ND - 1; ++j) {
                const double xj = x[j];
#pragma unroll
                for (int i = j + 1; i < ND; ++i) x[i] -= M2t[j * LD + i] * xj;
            }
#pragma unroll
            for (int j = ND - 1; j >= 0; --j) {
                x[j] *= rdM[j];
                const double xj = x[j];
#pragma unroll
                for (int i = 0; i < j; ++i) x[i] -= M2t[j * LD + i] * xj;
            }
        };
        double hx[NCR];
        if constexpr (NC > 0) {
            const double* Dh1 = sm + L::o_dh1;
            const double* Dh2t = sm + L::o_dh2t;
            const double* PJt = sm + L::o_pjt;
            const double* rdP = sm + L::o_rdp;
            const int* pivP = pivM + ND;
            solveM();
            double h[NC];
#pragma unroll
            for (int cc = 0; cc < NC; ++cc) h[cc] = tt == 3 ? Grow[jl.o_jk + cc * nk + it] : 0.0;
#pragma unroll
            for (int i = 0; i < ND; ++i) {
                const double yi = y[i], xi = x[i];
#pragma unroll
                for (int cc = 0; cc < NC; ++cc) { h[cc] += JCt[i * LP + cc] * yi; h[cc] += Dh2t[i * LP + cc] * xi; }
            }
#pragma unroll
            for (int cc = 0; cc < NC; ++cc) colh[cc * T] = h[cc];
#pragma unroll
            for (int i = 0; i < NC; ++i) hx[i] = colh[pivP[i] * T];
#pragma unroll
            for (int j = 0; j < NC - 1; ++j) {
                const double xj = hx[j];
#pragma unroll
                for (int i = j + 1; i < NC; ++i) hx[i] -= PJt[j * LP + i] * xj;
            }
#pragma unroll
            for (int j = NC - 1; j >= 0; --j) {
                hx[j] *= rdP[j];
                const double xj = hx[j];
#pragma unroll
                for (int i = 0; i < j; ++i) hx[i] -= PJt[j * LP + i] * xj;
            }
            // c + Dh1^T lambda_st
#pragma unroll
            for (int cc = 0; cc < NC; ++cc) {
                const double l = hx[cc];
#pragma unroll
                for (int j = 0; j < ND; ++j) c[j] += Dh1[cc * LD + j] * l;
            }
#pragma unroll
            for (int j = 0; j < ND; ++j) colc[j * T] = c[j];
        }
        solveM();   // q2_st
        // p2_st = D^2 p2 [xi_s, xi_t] + D2D2L2^T q2_st   (into c)
#pragma unroll
        for (int j = 0; j < ND; ++j) c[j] = rh ? rh[j * 4] : 0.0;
#pragma unroll
        for (int i = 0; i < ND; ++i) {
            const double yi = y[i], xi = x[i];
#pragma unroll
            for (int j = 0; j < ND; ++j) { c[j] += Hd[i * LD + j] * yi; c[j] += T22[i * LD + j] * xi; }
        }
        // ---- store (same indexing as d2_pair)
        const int kind = ts == 0 ? tt : (ts == 1 ? 3 + tt : (ts == 2 ? 5 + tt : 9));
        const bool mirror = (ts == tt) && (is != it);
        double* oq = p.out[0][kind];
        double* op = p.out[1][kind];
        double* ol = p.out[2][kind];
        const long base_q = (long)b * cnt_s * cnt_t;
        const long e1 = base_q + (long)is * cnt_t + it, e2 = base_q + (long)it * cnt_t + is;
        if (oq) {
#pragma unroll
            for (int j = 0; j < ND; ++j) oq[e1 * ND + j] = x[j];
            if (mirror) {
#pragma unroll
                for (int j = 0; j < ND; ++j) oq[e2 * ND + j] = x[j];
            }
        }
        if (op) {
#pragma unroll
            for (int j = 0; j < ND; ++j) op[e1 * ND + j] = c[j];
            if (mirror) {
#pragma unroll
                for (int j = 0; j < ND; ++j) op[e2 * ND + j] = c[j];
            }
        }
        if (p.z) {
            const double* z = sm + L::o_z;
            double acc = 0.0;
#pragma unroll
            for (int j = 0; j < ND; ++j) { acc += z[j] * x[j]; acc += z[nq + j] * c[j]; }
            const int nX = 2 * nq, nU = nu + nk;
            const bool sx = ts < 2, tx = tt < 2;
            const int xs = ts == 0 ? is : (ts == 1 ? nq + is : (ts == 2 ? is : nu + is));
            const int xt = tt == 0 ? it : (tt == 1 ? nq + it : (tt == 2 ? it : nu + it));
            if (sx && tx) {
                if (p.zxx) { p.zxx[((long)b * nX + xs) * nX + xt] = acc; p.zxx[((long)b * nX + xt) * nX + xs] = acc; }
            } else if (sx) {
                if (p.zxu) p.zxu[((long)b * nX + xs) * nU + xt] = acc;
            } else {
                if (p.zuu) { p.zuu[((long)b * nU + xs) * nU + xt] = acc; p.zuu[((long)b * nU + xt) * nU + xs] = acc; }
            }
        }
        if constexpr (NC > 0) {
            if (ol) {
#pragma unroll
                for (int cc = 0; cc < NC; ++cc) {
                    ol[e1 * NC + cc] = hx[cc];
                    if (mirror) ol[e2 * NC + cc] = hx[cc];
                }
            }
        }
    }
}

template <int ND, int NC>
cudaError_t d2solve_ct_run(cudaStream_t stream, const D2Params& p, const double* G, const JacLayout& jl, int nk, int nu,
                           long b0, long nb) {
    const size_t smem = D2Ct<ND, NC>::smem(ND + nk);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute((const void*)d2solve_ct_kernel<ND, NC>,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const int half = (p.nx + 1) / 2;
    d2solve_ct_kernel<ND, NC><<<(unsigned)(nb * half), kD2T, smem, stream>>>(p, G, jl, nk, nu, b0);
    return cudaGetLastError();
}

size_t d2solve_smem(int nd, int nk, int nc, int aux_size, int T) {
    return sizeof(double) * (size_t)(2 * nd * nd + 2 * nc * nd + aux_size + 2 * (nd + nk) + (3 * nd + 3 * nc) * T);
}

size_t d2jac_smem(int blob_bytes, int block, int nd, int nk) {
    const int n8 = ((blob_bytes + 7) / 8 + 1) & ~1;
    return sizeof(double) * ((size_t)n8 + (size_t)(block / 32) * 32 * 33) + (size_t)NzMaps::bytes(nd, nk);
}
cudaError_t d2jac_occupancy(bool varied, int block, size_t smem, int* blocks_per_sm, KernelInfo* info) {
    const void* fn = varied ? (const void*)d2jac_varied_kernel : (const void*)d2jac_kernel;
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, fn);
    if (e != cudaSuccess) return e;
    if (info) { info->regs = a.numRegs; info->max_threads = a.maxThreadsPerBlock; info->static_smem = a.sharedSizeBytes; info->local_bytes = a.localSizeBytes; }
    if (smem > 48 * 1024) {
        e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, fn, block, smem);
}
cudaError_t d2jac_run(const LaunchCfg& c, const WsStridedT<Dual>& w, const D2Params& p, double* G, const JacLayout& jl,
                      long b0, long nb, const VariedArgs* va) {
    const void* fn = va ? (const void*)d2jac_varied_kernel : (const void*)d2jac_kernel;
    if (c.smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c.smem);
        if (e != cudaSuccess) return e;
    }
    if (va) d2jac_varied_kernel<<<c.grid, c.block, c.smem, c.stream>>>(*c.sys, c.dblob, c.blob_bytes, w, p, G, jl, b0, nb, *va);
    else d2jac_kernel<<<c.grid, c.block, c.smem, c.stream>>>(*c.sys, c.dblob, c.blob_bytes, w, p, G, jl, b0, nb);
    return cudaGetLastError();
}
size_t d2solve_smem_needed(int nd, int nk, int nc, int nx, int aux_size) {
    if (nd == 22 && nc == 6) return D2Ct<22, 6>::smem(nd + nk);
    if (nd == 7 && nc == 4) return D2Ct<7, 4>::smem(nd + nk);
    return d2solve_smem(nd, nk, nc, aux_size, ((nx + 31) / 32) * 32);
}
cudaError_t d2solve_run(cudaStream_t stream, const D2Params& p, const double* G, const JacLayout& jl, int nd, int nk,
                        int nu, int nc, long b0, long nb) {
    // shapes with a compile-time-size pass B (the marionette of BASELINE.json's config 5)
    if (nd == 22 && nc == 6) return d2solve_ct_run<22, 6>(stream, p, G, jl, nk, nu, b0, nb);
    if (nd == 7 && nc == 4) return d2solve_ct_run<7, 4>(stream, p, G, jl, nk, nu, b0, nb);   // examples/pccd.py
    const int T = ((p.nx + 31) / 32) * 32;
    const size_t smem = d2solve_smem(nd, nk, nc, p.auxl.size, T);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute((const void*)d2solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    d2solve_kernel<<<(unsigned)(nb * p.nx), T, smem, stream>>>(p, G, jl, nd, nk, nu, nc, b0);
    return cudaGetLastError();
}

}  // namespace trepb
