// Second derivatives of the discrete flow (MidpointVI_calc_deriv2, trep/_trep/midpointvi.c:2516-2545):
//   q2, p2, lambda1  _d{q1q1, q1p1, q1u1, q1k2, p1p1, p1u1, p1k2, u1u1, u1k2, k2k2}
// in the reference's storage layout [wrt A][wrt B][output] (trep/_trep/trep.h:439-473).
//
// Formulation (not the reference's): with x = (q1, p1, u1, k2) the parameters and y = (q2_dyn,
// lambda) the unknowns of
//     F1 = p1 + D1L2(q1,q2) + fm2(q1,q2,u1) - Dh(q1)^T lambda = 0 ,   F2 = h(q2) = 0 ,
// the second-order implicit-function identity for a pair of parameters (s,t) is
//     F_y y_st + D^2F[xi_s, xi_t] = 0 ,   xi_s = (x_s, y_s)  the first-order tangent of deriv1,
// and  p2_st = D^2 H[xi_s, xi_t] + H_q2 q2_st  for  p2 = H = D2L2(q1,q2).
// D^2F[xi_s, xi_t] and D^2H[xi_s, xi_t] are obtained exactly by evaluating the first-order residual
// path of trepb_math.cuh on hyper-dual numbers (trepb_hd.h) along (xi_s, xi_t); the linear solve
// reuses deriv1's factorizations M2 = LU, proj = LU exactly as calc_deriv1 does for its right-hand
// sides (midpointvi.c:929-1098).  One thread per (instance, pair s<=t): the pairs of an instance are
// independent, which is the parallelism the reference spends its pthread row pool on
// (midpointvi.c:2536-2541).
#pragma once
// (included at the end of trepb_kernels.cuh)

namespace trepb {

struct AuxMat {
    const double* p; int ld;
    TREPB_HD double operator()(int i, int j) const { return p[i * ld + j]; }
};
struct AuxVec {
    const double* p;
    TREPB_HD double operator()(int i) const { return p[i]; }
};
// scratch vectors live in the v / a / b[0] components of hyper-dual workspace slots whose e1 e2k
// components hold the right-hand sides of the block (those are left untouched)
template <class Ws> struct FrV  { Ws* w; TREPB_HD double& operator()(int i) const { return w->fr(i).v; } };
template <class Ws> struct FrA  { Ws* w; TREPB_HD double& operator()(int i) const { return w->fr(i).a; } };
template <class Ws> struct FrB  { Ws* w; TREPB_HD double& operator()(int i) const { return w->fr(i).b[0]; } };
template <class Ws> struct HcV  { Ws* w; TREPB_HD double& operator()(int i) const { return w->hc(i).v; } };
template <class Ws> struct HcA  { Ws* w; TREPB_HD double& operator()(int i) const { return w->hc(i).a; } };

// type (0 q1, 1 p1, 2 u1, 3 k2) and index within the type of parameter s
TREPB_HD void split_param(int s, int nq, int nd, int nu, int* type, int* idx) {
    if (s < nq) { *type = 0; *idx = s; }
    else if (s < nq + nd) { *type = 1; *idx = s - nq; }
    else if (s < nq + nd + nu) { *type = 2; *idx = s - nq - nd; }
    else { *type = 3; *idx = s - nq - nd - nu; }
}
// number of direction blocks of an instance: for every s the parameters t = s .. nx-1 in blocks of N
TREPB_HD int d2_blocks(int nx, int N) {
    int n = 0;
    for (int s = 0; s < nx; ++s) n += (nx - s + N - 1) / N;
    return n;
}

// One (instance b, parameter s, block of nt <= N parameters t0 .. t0+nt-1 >= s): evaluates the residual
// once on hyper-duals carrying xi_s in e1 and xi_t in e2k, then solves and stores per pair.
template <class Sys, class Ws>
TREPB_HD void deriv2_block(const Sys& sys, Ws& ws, const D2Params& p, long b, int s, int t0, int nt) {
    using Real = typename Ws::Real;
    constexpr int N = (int)(sizeof(Real) / sizeof(double) - 2) / 2;
    const int nd = sys.ND(), nk = sys.NK(), nq = nd + nk, nu = sys.NU(), nc = sys.NC();
    int ts, is;
    split_param(s, nq, nd, nu, &ts, &is);
    const int cnt_s = ts == 0 ? nq : (ts == 1 ? nd : (ts == 2 ? nu : nk));
    const double* zs = p.q2_d[ts] + ((long)b * cnt_s + is) * nd;   // d q2_dyn / d s
    const double* ls = nc ? p.l1_d[ts] + ((long)b * cnt_s + is) * nc : nullptr;
    int tt[N], it[N], cnt_t[N];
    const double* zt[N];
    const double* lt[N];
    TREPB_HDU
    for (int k = 0; k < N; ++k) {
        const int t = t0 + (k < nt ? k : 0);
        split_param(t, nq, nd, nu, &tt[k], &it[k]);
        cnt_t[k] = tt[k] == 0 ? nq : (tt[k] == 1 ? nd : (tt[k] == 2 ? nu : nk));
        zt[k] = p.q2_d[tt[k]] + ((long)b * cnt_t[k] + it[k]) * nd;
        lt[k] = nc ? p.l1_d[tt[k]] + ((long)b * cnt_t[k] + it[k]) * nc : nullptr;
    }
    // ---- point z + e1 xi_s + sum_k e2k xi_tk   (unused directions k >= nt carry zero tangents)
    TREPB_UNROLL_SYS
    for (int i = 0; i < nq; ++i) {
        Real x1(p.q1[b * nq + i]), x2(p.q2[b * nq + i]);
        x1.a = (ts == 0 && is == i) ? 1.0 : 0.0;
        x2.a = i < nd ? zs[i] : ((ts == 3 && is == i - nd) ? 1.0 : 0.0);
        TREPB_HDU
        for (int k = 0; k < N; ++k) {
            const bool on = k < nt;
            x1.b[k] = (on && tt[k] == 0 && it[k] == i) ? 1.0 : 0.0;
            x2.b[k] = !on ? 0.0 : (i < nd ? zt[k][i] : ((tt[k] == 3 && it[k] == i - nd) ? 1.0 : 0.0));
        }
        ws.q1(i) = x1;
        ws.q2(i) = x2;
    }
    TREPB_UNROLL_SYS
    for (int i = 0; i < nu; ++i) {
        Real x(p.u1[b * nu + i]);
        x.a = (ts == 2 && is == i) ? 1.0 : 0.0;
        TREPB_HDU for (int k = 0; k < N; ++k) x.b[k] = (k < nt && tt[k] == 2 && it[k] == i) ? 1.0 : 0.0;
        ws.u1(i) = x;
    }
    TREPB_UNROLL_SYS
    for (int i = 0; i < nc; ++i) {
        Real x(p.lam[b * nc + i]);
        x.a = ls[i];
        TREPB_HDU for (int k = 0; k < N; ++k) x.b[k] = k < nt ? lt[k][i] : 0.0;
        ws.lam(i) = x;
    }
    const double t1 = p.t1 ? p.t1[b] : p.t1s;
    const double t2 = p.t2 ? p.t2[b] : (t1 + p.dts);
    const double dt = t2 - t1;
    // ---- residual along the tangents (same call sequence as calc_f, midpointvi.c:533-565)
    if (nc > 0) {
        set_point(sys, ws, 1, dt);
        pass1(sys, ws, false, true);
        constraints_eval(sys, ws, 2, 1);
    }
    eval_mid(sys, ws, dt, 1);
    TREPB_UNROLL_SYS
    for (int j = 0; j < nd; ++j) {
        Real f = (0.5 * dt * ws.Lq(j) - ws.Lv(j)) + dt * ws.Fo(j);
        TREPB_UNROLL_SYS
        for (int cc = 0; cc < nc; ++cc) f -= ws.Dh1(cc, j) * ws.lam(cc);
        const Real h2 = 0.5 * dt * ws.Lq(j) + ws.Lv(j);
        ws.fr(j) = f;      // .ab[k] = R1 of pair k
        ws.p2(j) = h2;     // .ab[k] = D^2 H [xi_s, xi_tk]
    }
    if (nc > 0) {
        set_point(sys, ws, 2, dt);
        pass1(sys, ws, false, true);
        constraints_eval(sys, ws, 1, 2);   // hc(cc).ab[k] = R2 of pair k
    }
    // ---- per pair: solve (calc_deriv1's scheme): lambda_st = proj^-1 (Dh2 M2^-1 c + R2),
    //      q2_st = M2^-1 (c + Dh1^T lambda_st),  p2_st = D^2H + D2D2L2^T q2_st
    const double* aux = p.aux + (long)b * p.auxl.size;
    const AuxMat M2{aux + p.auxl.o_m2, nd}, PJ{aux + p.auxl.o_pj, nc}, T22{aux + p.auxl.o_t22, nd};
    const AuxMat Dh1{aux + p.auxl.o_dh1, nd}, Dh2{aux + p.auxl.o_dh2, nd};
    const AuxVec M2p{aux + p.auxl.o_m2p}, PJp{aux + p.auxl.o_pjp};
    TREPB_HDU
    for (int k = 0; k < N; ++k) {
        if (k >= nt) continue;
        TREPB_UNROLL_SYS
        for (int j = 0; j < nd; ++j) { const double c = -ws.fr(j).ab[k]; ws.fr(j).v = c; ws.fr(j).a = c; }   // tnd = col = c = -R1
        if (nc > 0) {
            lu_solve<Sys>(M2, nd, M2p, FrV<Ws>{&ws}, FrB<Ws>{&ws});
            TREPB_UNROLL_SYS
            for (int cc = 0; cc < nc; ++cc) {
                double sacc = 0.0;
                TREPB_UNROLL_SYS
                for (int j = 0; j < nd; ++j) sacc += Dh2(cc, j) * ws.fr(j).v;
                ws.hc(cc).v = sacc + ws.hc(cc).ab[k];
            }
            lu_solve<Sys>(PJ, nc, PJp, HcV<Ws>{&ws}, HcA<Ws>{&ws});
            TREPB_UNROLL_SYS
            for (int j = 0; j < nd; ++j) {
                double sacc = ws.fr(j).a;
                TREPB_UNROLL_SYS
                for (int cc = 0; cc < nc; ++cc) sacc += Dh1(cc, j) * ws.hc(cc).v;
                ws.fr(j).a = sacc;
            }
        }
        lu_solve<Sys>(M2, nd, M2p, FrA<Ws>{&ws}, FrB<Ws>{&ws});
        // ---- store: kind index of (type s <= type t)
        const int kind = ts == 0 ? tt[k] : (ts == 1 ? 3 + tt[k] : (ts == 2 ? 5 + tt[k] : 9));
        const bool mirror = (ts == tt[k]) && (is != it[k]);
        double* oq = p.out[0][kind];
        double* op = p.out[1][kind];
        double* ol = p.out[2][kind];
        const long base_q = (long)b * cnt_s * cnt_t[k];
        const long e1 = base_q + (long)is * cnt_t[k] + it[k], e2 = base_q + (long)it[k] * cnt_t[k] + is;
        double acc = 0.0;
        const double* z = p.z ? p.z + (long)b * 2 * nq : nullptr;
        TREPB_UNROLL_SYS
        for (int j = 0; j < nd; ++j) {
            const double qv = ws.fr(j).a;
            double pv = ws.p2(j).ab[k];
            TREPB_UNROLL_SYS
            for (int kk = 0; kk < nd; ++kk) pv += T22(kk, j) * ws.fr(kk).a;
            if (oq) {
                oq[e1 * nd + j] = qv;
                if (mirror) oq[e2 * nd + j] = qv;
            }
            if (op) {
                op[e1 * nd + j] = pv;
                if (mirror) op[e2 * nd + j] = pv;
            }
            if (z) acc += z[j] * qv + z[nq + j] * pv;
        }
        if (z) {
            // z-contraction in the DSystem layout: X = [Q; p; v], U = [u; rho]  (dsystem.py:320-386)
            const int nX = 2 * nq, nU = nu + nk;
            const bool sx = ts < 2, tx = tt[k] < 2;
            const int xs = ts == 0 ? is : (ts == 1 ? nq + is : (ts == 2 ? is : nu + is));
            const int xt = tt[k] == 0 ? it[k] : (tt[k] == 1 ? nq + it[k] : (tt[k] == 2 ? it[k] : nu + it[k]));
            if (sx && tx) {
                if (p.zxx) { p.zxx[((long)b * nX + xs) * nX + xt] = acc; p.zxx[((long)b * nX + xt) * nX + xs] = acc; }
            } else if (sx) {
                if (p.zxu) p.zxu[((long)b * nX + xs) * nU + xt] = acc;
            } else {
                if (p.zuu) { p.zuu[((long)b * nU + xs) * nU + xt] = acc; p.zuu[((long)b * nU + xt) * nU + xs] = acc; }
            }
        }
        if (ol) {
            TREPB_UNROLL_SYS
            for (int cc = 0; cc < nc; ++cc) {
                const double lv = ws.hc(cc).v;
                ol[e1 * nc + cc] = lv;
                if (mirror) ol[e2 * nc + cc] = lv;
            }
        }
    }
}

#if defined(__CUDACC__)
template <class Sys, bool S = Sys::kStatic>
struct CtxHD;
template <class Sys>
struct CtxHD<Sys, true> {
    Sys sys;
    WsStatic<Sys, HD> ws;
    __device__ __forceinline__ CtxHD(const RtSys&, const char*, int, const WsStridedT<HDG>&, long, long,
                                     const typename Sys::Params& par) { sys.par = par; }
};
template <class Sys>
struct CtxHD<Sys, false> {
    RtSys sys;
    WsStridedT<HDG> ws;
    __device__ __forceinline__ CtxHD(const RtSys& s, const char* dblob, int blob_bytes, const WsStridedT<HDG>& w,
                                     long tid, long nthreads, const typename Sys::Params&) {
        extern __shared__ double smem_[];
        const int n8 = (blob_bytes + 7) / 8;
        const double* src = (const double*)dblob;
        for (int i = threadIdx.x; i < n8; i += blockDim.x) smem_[i] = src[i];
        __syncthreads();
        sys = s.rebased(dblob, (const char*)smem_);
        ws = w;
        ws.base = w.base + tid;
        ws.stride = (unsigned)nthreads;
    }
};

// kVaried: work item (b, s, block of t) runs on row b of the per-instance parameters.  The items of one instance land
// on different threads, so each item loads its row (load_params, trepb_kernels.cuh).
template <class Sys, bool kVaried>
__device__ __forceinline__ void
d2_body(const RtSys& rsys, const char* dblob, int blob_bytes, const WsStridedT<HDG>& wsp, const D2Params& p,
        const typename Sys::Params& par, const VariedArgs& va) {
    const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long nth = (long)gridDim.x * blockDim.x;
    CtxHD<Sys> c(rsys, dblob, blob_bytes, wsp, tid, nth, par);
    auto& sys = c.sys;
    auto& ws = c.ws;
    using Ws = typename std::remove_reference<decltype(ws)>::type;
    const int nd = sys.ND(), nk = sys.NK(), nq = nd + nk, nu = sys.NU(), nc = sys.NC();
    // work item = (instance, parameter s, block of N parameters t >= s); N = directions per hyper-dual
    // number of this kernel's workspace type (trepb_hd.h)
    constexpr int N = (int)(sizeof(typename Ws::Real) / sizeof(double) - 2) / 2;
    const int nblk = d2_blocks(p.nx, N);
    const long total = p.batch * (long)nblk;
    for (long g = tid; g < total; g += nth) {
        const long b = g / nblk;
        if (p.status && p.status[b] != 0) continue;
        load_params<Sys, kVaried>(c, va, b, tid);
        int pr = (int)(g - b * nblk), s = 0;
        for (;;) {
            const int nb = (p.nx - s + N - 1) / N;
            if (pr < nb) break;
            pr -= nb;
            ++s;
        }
        const int t0 = s + pr * N;
        const int nt = p.nx - t0 < N ? p.nx - t0 : N;
        deriv2_block(sys, ws, p, b, s, t0, nt);
    }
}

template <class Sys>
__global__ void __launch_bounds__(128)
d2_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStridedT<HDG> wsp, const D2Params p,
          const typename Sys::Params par) {
    d2_body<Sys, false>(rsys, dblob, blob_bytes, wsp, p, par, VariedArgs{});
}
template <class Sys>
__global__ void __launch_bounds__(128)
d2_varied_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStridedT<HDG> wsp, const D2Params p,
                 const VariedArgs va) {
    d2_body<Sys, true>(rsys, dblob, blob_bytes, wsp, p, typename Sys::Params{}, va);
}

template <class Sys>
struct LaunchersD2 {
    // d2_kernel for plain launches, d2_varied_kernel for per-instance parameters
    static cudaError_t run(const LaunchCfg& c, const WsStridedT<HDG>& w, const D2Params& p, const VariedArgs* va) {
        RtSys rs{};
        if (c.sys) rs = *c.sys;
        const void* fn = va ? (const void*)d2_varied_kernel<Sys> : (const void*)d2_kernel<Sys>;
        cudaError_t e = Launchers<Sys>::prep(fn, c.smem);
        if (e != cudaSuccess) return e;
        if (va) d2_varied_kernel<Sys><<<c.grid, c.block, c.smem, c.stream>>>(rs, c.dblob, c.blob_bytes, w, p, *va);
        else d2_kernel<Sys><<<c.grid, c.block, c.smem, c.stream>>>(rs, c.dblob, c.blob_bytes, w, p, Launchers<Sys>::spec_params(c));
        return cudaGetLastError();
    }
    static cudaError_t occupancy(bool varied, int block, size_t smem, int* blocks_per_sm, KernelInfo* info) {
        return Launchers<Sys>::occupancy_of(varied ? (const void*)d2_varied_kernel<Sys> : (const void*)d2_kernel<Sys>,
                                            block, smem, blocks_per_sm, info);
    }
};
#endif

}  // namespace trepb
