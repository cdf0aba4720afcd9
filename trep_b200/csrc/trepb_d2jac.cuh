// Second derivatives of the discrete flow for table-driven systems, in O(nx) evaluations per
// instance (MidpointVI_calc_deriv2, trep/_trep/midpointvi.c:2516-2545; same outputs and layout as
// trepb_d2.cuh, a different factorisation of the work).
//
// With z = (q1, q2, u1, lambda), parameters x = (q1, p1, u1, k2), first-order tangents
// xi_s = (x_s, y_s) from deriv1 and the residual  F = (F1, F2) = (p1 + D1L2 + fm2 - Dh(q1)^T lambda,
// h(q2)),  the bilinear form the implicit-function identity needs is
//     D^2F[xi_s, xi_t] = ( d/de  J(z + e xi_s) |_{e=0} ) xi_t ,        J = dF/dz ,
// i.e. the directional derivative of the JACOBIAN tables along xi_s, applied to xi_t.  J is what the
// linearize kernels already assemble (calc_deriv1_cache, midpointvi.c:749-861: D1D1L2, D2D1L2,
// D1D2L2, D2D2L2, the force derivatives, Dh(q1), Dh(q2), sum_c lambda_c DDh_c(q1)).  So:
//
//   pass A  (d2jac_kernel, one thread per (instance, s)):  evaluate the second-order table path of
//           trepb_math.cuh ONCE on dual numbers v + a e along xi_s and write the e-parts of the
//           table combinations (JacLayout) - nx evaluations per instance instead of the
//           nx (nx + 1) / 2 hyper-dual residual evaluations of trepb_d2.cuh (80 vs 3240 for the
//           marionette);
//   pass B  (d2solve_kernel, one CTA per (instance, s), one thread per t >= s):  contract with xi_t
//           (unit rows + a dense nd x (nd + nc) product from shared memory), solve with deriv1's
//           factors M2 = LU, proj = LU exactly as calc_deriv1 does for its right-hand sides
//           (midpointvi.c:929-1098), store the tensors and / or their z-contraction.
//
// The reference hand-expands third-order tables instead (calc_deriv2_cache_*,
// midpointvi.c:1122-1532, on system.c:204-268, 336-393, 514-557); nothing of that is transcribed.
#pragma once
#include <math.h>
#include "trepb_sys.h"

namespace trepb {

// ---------------------------------------------------------------------------------------------
// dual numbers  v + a e ,  e^2 = 0
// ---------------------------------------------------------------------------------------------
struct Dual {
    double v, a;
    Dual() = default;
    TREPB_HD Dual(double x) : v(x), a(0.0) {}
    TREPB_HD Dual(double x, double d) : v(x), a(d) {}
};
TREPB_HD Dual operator-(const Dual& x) { return Dual(-x.v, -x.a); }
TREPB_HD Dual operator+(const Dual& x, const Dual& y) { return Dual(x.v + y.v, x.a + y.a); }
TREPB_HD Dual operator-(const Dual& x, const Dual& y) { return Dual(x.v - y.v, x.a - y.a); }
TREPB_HD Dual operator*(const Dual& x, const Dual& y) { return Dual(x.v * y.v, x.a * y.v + x.v * y.a); }
TREPB_HD Dual operator+(const Dual& x, double y) { return Dual(x.v + y, x.a); }
TREPB_HD Dual operator+(double y, const Dual& x) { return Dual(x.v + y, x.a); }
TREPB_HD Dual operator-(const Dual& x, double y) { return Dual(x.v - y, x.a); }
TREPB_HD Dual operator-(double y, const Dual& x) { return Dual(y - x.v, -x.a); }
TREPB_HD Dual operator*(const Dual& x, double y) { return Dual(x.v * y, x.a * y); }
TREPB_HD Dual operator*(double y, const Dual& x) { return Dual(x.v * y, x.a * y); }
TREPB_HD Dual du_inv(const Dual& y) { const double r = 1.0 / y.v; return Dual(r, -r * r * y.a); }
TREPB_HD Dual operator/(const Dual& x, const Dual& y) { return x * du_inv(y); }
TREPB_HD Dual operator/(double x, const Dual& y) { return x * du_inv(y); }
TREPB_HD Dual operator/(const Dual& x, double y) { return x * (1.0 / y); }
TREPB_HD Dual& operator+=(Dual& x, const Dual& y) { x.v += y.v; x.a += y.a; return x; }
TREPB_HD Dual& operator-=(Dual& x, const Dual& y) { x.v -= y.v; x.a -= y.a; return x; }
TREPB_HD Dual& operator*=(Dual& x, const Dual& y) { x = x * y; return x; }
TREPB_HD Dual& operator+=(Dual& x, double y) { x.v += y; return x; }
TREPB_HD Dual& operator-=(Dual& x, double y) { x.v -= y; return x; }
TREPB_HD Dual& operator*=(Dual& x, double y) { x.v *= y; x.a *= y; return x; }
TREPB_HD void sincos_(double x, double* s, double* c);   // trepb_math.cuh
TREPB_HD void sincos_(const Dual& x, Dual* s, Dual* c) {
    double sn, cs;
    sincos_(x.v, &sn, &cs);
    *s = Dual(sn, cs * x.a);
    *c = Dual(cs, -sn * x.a);
}
TREPB_HD Dual sqrt_(const Dual& x) { const double r = sqrt(x.v); return Dual(r, 0.5 / r * x.a); }
TREPB_HD bool isnan_(const Dual& x) { return isnan(x.v); }

// ---------------------------------------------------------------------------------------------
// what pass A hands to pass B, per (instance, s):  e-parts of the Jacobian tables along xi_s
//   Q  [nq][nd][4]  for (i, j):  0  JA = d F1_j / d q1_i   (D1 of the residual incl. -sum_c lambda_c DDh_c)
//                                1  JB = d F1_j / d q2_i   (rows i >= nd are the kinematic configs k2)
//                                2  HA = d p2_j / d q1_i
//                                3  HB = d p2_j / d q2_i
//                   (interleaved: pass A forms the four combinations from one read of the tables)
//   JU [nu][nd]   d F1_j / d u1_i
//   JL [nc][nd]   d F1_j / d lambda_c    ( = -Dh(q1) )
//   JC [nc][nd]   d F2_c / d q2_i , i dynamic        JK [nc][nk]  the same for the kinematic configs
// ---------------------------------------------------------------------------------------------
struct JacLayout {
    int o_q, o_ju, o_jl, o_jc, o_jk, size;
    TREPB_HD void set(int nd, int nk, int nu, int nc) {
        const int nq = nd + nk;
        int o = 0;
        o_q = o; o += 4 * nq * nd;
        o_ju = o; o += nu * nd;
        o_jl = o; o += nc * nd;
        o_jc = o; o += nc * nd;
        o_jk = o; o += nc * nk;
        size = o;
    }
    TREPB_HD int q(int i, int j, int nd, int w) const { return o_q + (i * nd + j) * 4 + w; }
};

}  // namespace trepb

#include "trepb_math.cuh"
#include "trepb_kernels.cuh"

namespace trepb {

// ---- structure of the second-order tables: which entries can be non-zero (supersets).  Pass A
// clears and reads only those; for the marionette that is 1/5 of the 40 x 40 entries.
//   L [nq][nq]  Lqq / Lvq / Lvv : two configs on one chain (system.c:170-180 skips the rest too),
//               a ConfigSpring's diagonal entry, the dependent configs of a LinearSpring
//   F [nd][nq]  Fq / Fv         : Damping's diagonal, the dependent configs of a LinearDamper
//   H [nq][nq]  sum_c lambda_c DDh_c : pairs of configs one constraint depends on
struct NzMaps {
    uint8_t *L, *F, *H;
    TREPB_HD static int bytes(int nd, int nk) { const int nq = nd + nk; return ((2 * nq * nq + nd * nq) + 7) & ~7; }
    TREPB_HD void place(uint8_t* base, int nd, int nk) { const int nq = nd + nk; L = base; H = L + nq * nq; F = H + nq * nq; }
};
template <class Sys>
TREPB_HD void d2jac_build_nz(const Sys& sys, const NzMaps& nz, int lane, int nlanes) {
    const int nd = sys.ND(), nq = sys.NQ();
    for (int e = lane; e < nq * nq; e += nlanes) {
        const int i = e / nq, j = e - i * nq;
        const int Fi = sys.cfg_frame(i), Fj = sys.cfg_frame(j);
        bool l = (Fj >= 0 && sys.dep(Fj, i)) || (Fi >= 0 && sys.dep(Fi, j));
        for (int p = 0; p < sys.NPOT(); ++p) {
            const int kind = sys.pot_kind(p);
            if (kind == P_CONFIG_SPRING || kind == P_NONLINEAR_CONFIG_SPRING) l = l || (i == j && i == sys.pot_i(p, 0));
            else if (kind == P_LINEAR_SPRING) {
                const int A = sys.pot_i(p, 0), B = sys.pot_i(p, 1);
                l = l || ((sys.dep(A, i) || sys.dep(B, i)) && (sys.dep(A, j) || sys.dep(B, j)));
            }
        }
        nz.L[e] = l ? 1 : 0;
        bool h = false;
        for (int c = 0; c < sys.NC(); ++c) {
            const int A = sys.con_i(c, 0), B = sys.con_i(c, 1);
            const int third = sys.con_kind(c) == C_DISTANCE ? sys.con_i(c, 2) : -1;
            h = h || ((sys.dep(A, i) || sys.dep(B, i) || third == i) && (sys.dep(A, j) || sys.dep(B, j) || third == j));
        }
        nz.H[e] = h ? 1 : 0;
        if (i < nd) {
            bool f = false;
            for (int fo = 0; fo < sys.NFORCE(); ++fo) {
                const int kind = sys.force_kind(fo);
                if (kind == F_DAMPING) f = f || i == j;
                else if (kind == F_LINEAR_DAMPER) {
                    const int off = sys.force_i(fo, 0);
                    const int A = sys.ipool(off), B = sys.ipool(off + 1);
                    f = f || ((sys.dep(A, i) || sys.dep(B, i)) && (sys.dep(A, j) || sys.dep(B, j)));
                } else if (kind == F_BODY_WRENCH || kind == F_HYBRID_WRENCH || kind == F_SPATIAL_WRENCH) {
                    const int A = sys.force_i(fo, 0);
                    f = f || (sys.dep(A, i) && sys.dep(A, j));
                }
            }
            nz.F[i * nq + j] = f ? 1 : 0;
        }
    }
}

// ---- pass A, evaluation: the tables of calc_deriv1_cache at z + e xi_s  (left in ws)
template <class Sys, class Ws>
TREPB_HD void d2jac_eval(const Sys& sys, Ws& ws, const NzMaps& nz, const D2Params& p, long b, int s) {
    using Real = typename Ws::Real;
    const int nd = sys.ND(), nk = sys.NK(), nq = nd + nk, nu = sys.NU(), nc = sys.NC();
    int ts, is;
    split_param(s, nq, nd, nu, &ts, &is);
    const int cnt_s = ts == 0 ? nq : (ts == 1 ? nd : (ts == 2 ? nu : nk));
    const double* zs = p.q2_d[ts] + ((long)b * cnt_s + is) * nd;   // d q2_dyn / d s
    const double* ls = nc ? p.l1_d[ts] + ((long)b * cnt_s + is) * nc : nullptr;
    for (int i = 0; i < nq; ++i) {
        ws.q1(i) = Real(p.q1[b * nq + i], (ts == 0 && is == i) ? 1.0 : 0.0);
        ws.q2(i) = Real(p.q2[b * nq + i], i < nd ? zs[i] : ((ts == 3 && is == i - nd) ? 1.0 : 0.0));
    }
    for (int i = 0; i < nu; ++i) ws.u1(i) = Real(p.u1[b * nu + i], (ts == 2 && is == i) ? 1.0 : 0.0);
    for (int i = 0; i < nc; ++i) ws.lam(i) = Real(p.lam[b * nc + i], ls[i]);
    const double t1 = p.t1 ? p.t1[b] : p.t1s;
    const double t2 = p.t2 ? p.t2[b] : (t1 + p.dts);
    const double dt = t2 - t1;
    // clear the table entries that can be written
    for (int i = 0; i < nq; ++i)
        for (int j = 0; j < nq; ++j) {
            if (nz.L[i * nq + j]) { ws.Lqq(i, j) = 0.0; ws.Lvq(i, j) = 0.0; ws.Lvv(i, j) = 0.0; }
            if (nc > 0 && nz.H[i * nq + j]) ws.DDhl(i, j) = 0.0;
        }
    for (int j = 0; j < nd; ++j) {
        for (int i = 0; i < nq; ++i)
            if (nz.F[j * nq + i]) { ws.Fq(j, i) = 0.0; ws.Fv(j, i) = 0.0; }
        for (int u = 0; u < nu; ++u) ws.Fu(j, u) = 0.0;
    }
    if (nc > 0) {
        set_point(sys, ws, 1, dt);
        pass1(sys, ws, false, true);
        constraints_eval(sys, ws, 2 | 4, 1, false);   // Dh1, DDhl = sum_c lambda_c DDh_c(q1)
        set_point(sys, ws, 2, dt);
        pass1(sys, ws, false, true);
        constraints_eval(sys, ws, 2, 2);              // Dh2
    }
    // eval_mid(order 2) with the table clearing done above
    set_point(sys, ws, 0, dt);
    pass1(sys, ws, true, sys.pairs_mid());   // world poses at the midpoint only for springs / dampers
    pass2(sys, ws, 2, false);
    add_potentials(sys, ws, 2);
    forces_eval(sys, ws, 2, false);
}

// ---- pass A, output: e-parts of the table combinations, pushed in JacLayout order
template <class Sys, class Ws, class Sink>
TREPB_HD void d2jac_emit(const Sys& sys, Ws& ws, const NzMaps& nz, double dt, Sink& out) {
    const int nd = sys.ND(), nk = sys.NK(), nq = nd + nk, nu = sys.NU(), nc = sys.NC();
    // the four combinations of calc_deriv1_cache (trepb_math.cuh deriv1, midpointvi.c:771-858)
    for (int a = 0; a < nq; ++a) {
        for (int b = 0; b < nd; ++b) {
            double qq = 0.0, vv = 0.0, vab = 0.0, vba = 0.0, fq = 0.0, fv = 0.0;
            if (nz.L[a * nq + b]) {
                qq = 0.25 * dt * ws.Lqq(a, b).a; vv = 1.0 / dt * ws.Lvv(a, b).a;
                vab = 0.5 * ws.Lvq(a, b).a; vba = 0.5 * ws.Lvq(b, a).a;
            }
            if (nz.F[b * nq + a]) { fq = 0.5 * dt * ws.Fq(b, a).a; fv = ws.Fv(b, a).a; }
            double ja = (qq + vv) - vab - vba + (fq - fv);
            if (nc > 0 && nz.H[a * nq + b]) ja -= ws.DDhl(a, b).a;
            out.push(ja);
            out.push((qq - vv) + vab - vba + (fq + fv));
            out.push((qq - vv) - vab + vba);
            out.push((qq + vv) + vab + vba);
        }
    }
    for (int u = 0; u < nu; ++u)
        for (int j = 0; j < nd; ++j) out.push(dt * ws.Fu(j, u).a);
    for (int c = 0; c < nc; ++c)
        for (int j = 0; j < nd; ++j) out.push(-ws.Dh1(c, j).a);
    for (int c = 0; c < nc; ++c)
        for (int j = 0; j < nd; ++j) out.push(ws.Dh2(c, j).a);
    for (int c = 0; c < nc; ++c)
        for (int k = 0; k < nk; ++k) out.push(ws.Dh2(c, nd + k).a);
}

// ---- pass B, one pair (s, t):  contraction with xi_t, solves, stores.
// Shared by every pair of (instance, s): Jd = JB rows < nd, Hd = HB rows < nd, JL, JC (pointers may
// be shared memory); Grow = the whole JacLayout record (for the single rows a pair picks);
// aux = deriv1's factors (AuxLayout).  Per-pair vectors y (nd), lt (nc), c (nd), x (nd), h (nc),
// hx (nc) are addressed with stride vs (column per thread in shared memory on the device).
struct D2Pair {
    const double *Jd, *Hd, *JL, *JC, *Grow, *aux, *z;
    JacLayout jl;
    AuxLayout al;
};
TREPB_HD void d2_lu_apply(const double* A, int n, const double* piv, const double* b, double* x, int vs) {
    // x = (LU)^-1 P b with lu_decomp's storage (math-code.c:434-461)
    for (int i = 0; i < n; ++i) {
        double t = b[(int)piv[i] * vs];
        for (int j = 0; j < i; ++j) t -= A[i * n + j] * x[j * vs];
        x[i * vs] = t;
    }
    for (int i = n - 1; i >= 0; --i) {
        double t = x[i * vs];
        for (int j = i + 1; j < n; ++j) t -= A[i * n + j] * x[j * vs];
        x[i * vs] = t / A[i * n + i];
    }
}
TREPB_HD void d2_pair(const D2Pair& P, const D2Params& p, long b, int nd, int nk, int nu, int nc, int s, int t,
                      double* y, double* lt, double* c, double* x, double* h, double* hx, int vs) {
    const int nq = nd + nk;
    int ts, is, tt, it;
    split_param(s, nq, nd, nu, &ts, &is);
    split_param(t, nq, nd, nu, &tt, &it);
    const int cnt_s = ts == 0 ? nq : (ts == 1 ? nd : (ts == 2 ? nu : nk));
    const int cnt_t = tt == 0 ? nq : (tt == 1 ? nd : (tt == 2 ? nu : nk));
    {
        const double* zt = p.q2_d[tt] + ((long)b * cnt_t + it) * nd;
        for (int i = 0; i < nd; ++i) y[i * vs] = zt[i];
        if (nc) {
            const double* l = p.l1_d[tt] + ((long)b * cnt_t + it) * nc;
            for (int cc = 0; cc < nc; ++cc) lt[cc * vs] = l[cc];
        }
    }
    // single rows this t picks: its own unit component of xi_t
    const double* r1 = tt == 0 ? P.Grow + P.jl.q(it, 0, nd, 0)
                     : tt == 2 ? P.Grow + P.jl.o_ju + it * nd
                     : tt == 3 ? P.Grow + P.jl.q(nd + it, 0, nd, 1) : nullptr;
    const double* rh = tt == 0 ? P.Grow + P.jl.q(it, 0, nd, 2)
                     : tt == 3 ? P.Grow + P.jl.q(nd + it, 0, nd, 3) : nullptr;
    const int r1s = tt == 2 ? 1 : 4;
    // c = -R1 ,  R1 = D^2 F1 [xi_s, xi_t]
    for (int j = 0; j < nd; ++j) {
        double acc = r1 ? r1[j * r1s] : 0.0;
        for (int i = 0; i < nd; ++i) acc += P.Jd[i * nd + j] * y[i * vs];
        for (int cc = 0; cc < nc; ++cc) acc += P.JL[cc * nd + j] * lt[cc * vs];
        c[j * vs] = -acc;
    }
    const double* M2 = P.aux + P.al.o_m2;
    const double* M2p = P.aux + P.al.o_m2p;
    if (nc > 0) {
        const double* PJ = P.aux + P.al.o_pj;
        const double* PJp = P.aux + P.al.o_pjp;
        const double* Dh1 = P.aux + P.al.o_dh1;
        const double* Dh2 = P.aux + P.al.o_dh2;
        d2_lu_apply(M2, nd, M2p, c, x, vs);
        for (int cc = 0; cc < nc; ++cc) {
            // R2 = D^2 F2 [xi_s, xi_t]
            double acc = tt == 3 ? P.Grow[P.jl.o_jk + cc * nk + it] : 0.0;
            for (int i = 0; i < nd; ++i) acc += P.JC[cc * nd + i] * y[i * vs];
            for (int j = 0; j < nd; ++j) acc += Dh2[cc * nd + j] * x[j * vs];
            h[cc * vs] = acc;
        }
        d2_lu_apply(PJ, nc, PJp, h, hx, vs);   // lambda_st
        for (int j = 0; j < nd; ++j) {
            double acc = c[j * vs];
            for (int cc = 0; cc < nc; ++cc) acc += Dh1[cc * nd + j] * hx[cc * vs];
            c[j * vs] = acc;
        }
    }
    d2_lu_apply(M2, nd, M2p, c, x, vs);        // q2_st
    // ---- store (layout [wrt A][wrt B][out], trep.h:439-473; same indexing as trepb_d2.cuh)
    const double* T22 = P.aux + P.al.o_t22;
    const int kind = ts == 0 ? tt : (ts == 1 ? 3 + tt : (ts == 2 ? 5 + tt : 9));
    const bool mirror = (ts == tt) && (is != it);
    double* oq = p.out[0][kind];
    double* op = p.out[1][kind];
    double* ol = p.out[2][kind];
    const long base_q = (long)b * cnt_s * cnt_t;
    const long e1 = base_q + (long)is * cnt_t + it, e2 = base_q + (long)it * cnt_t + is;
    double acc = 0.0;
    const double* z = P.z;
    for (int j = 0; j < nd; ++j) {
        const double qv = x[j * vs];
        double pv = rh ? rh[j * 4] : 0.0;   // D^2 p2 [xi_s, xi_t] ...
        for (int i = 0; i < nd; ++i) pv += P.Hd[i * nd + j] * y[i * vs];
        for (int k = 0; k < nd; ++k) pv += T22[k * nd + j] * x[k * vs];   // ... + D2D2L2^T q2_st
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
    if (ol) {
        for (int cc = 0; cc < nc; ++cc) {
            const double lv = hx[cc * vs];
            ol[e1 * nc + cc] = lv;
            if (mirror) ol[e2 * nc + cc] = lv;
        }
    }
}

#if defined(__CUDACC__)
// launchers (trepb_d2jac.cu)
// pass A: d2jac_kernel, or d2jac_varied_kernel for a non-null VariedArgs / `varied` (table-driven map and slots)
cudaError_t d2jac_occupancy(bool varied, int block, size_t smem, int* blocks_per_sm, KernelInfo* info);
size_t d2jac_smem(int blob_bytes, int block, int nd, int nk);
cudaError_t d2jac_run(const LaunchCfg& c, const WsStridedT<Dual>& w, const D2Params& p, double* G, const JacLayout& jl,
                      long b0, long nb, const VariedArgs* va);
size_t d2solve_smem(int nd, int nk, int nc, int aux_size, int T);
// shared memory pass B needs for this shape (compile-time-size flavour where one exists)
size_t d2solve_smem_needed(int nd, int nk, int nc, int nx, int aux_size);
cudaError_t d2solve_run(cudaStream_t stream, const D2Params& p, const double* G, const JacLayout& jl, int nd, int nk,
                        int nu, int nc, long b0, long nb);
#endif

}  // namespace trepb
