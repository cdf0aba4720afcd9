// Link-level ("articulated body") view of a flattened system for the team-cooperative kernels
// (trepb_coop_math.cuh): one warp works on one instance, its workspace lives in shared memory.
//
// The frame tree of the description (trep/system.py:733-771, trep/frame.py:658-721) is condensed
// on the host, once per system:
//   * every frame driven by a config becomes a LINK; the constant frames between two links are
//     multiplied into one constant pre-transform (Rc, pc) of the lower link;
//   * the masses that hang off a link through constant frames are summed into one rigid-body
//     inertia (m, h = m c, Ibar about the link origin) of that link;
//   * the frames used by constraints become POINTS: a link index and a constant offset;
//   * links are numbered level by level (all links with k variable ancestors before those with
//     k+1), so one tree level is a contiguous index range and the children of a link are
//     contiguous too;
//   * the (ancestor, descendant) link pairs that carry non-zero entries of the second-order
//     Lagrangian tables (system.c:129-557: L_dqdq, L_ddqdq, L_ddqddq are zero unless both configs
//     lie on one chain) are enumerated, with a config x config map into that list.
//
// The arithmetic built on these tables is the same mathematics as the reference's frame caches,
// evaluated in world ("spatial") coordinates - see trepb_coop_math.cuh.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../include/trepb.h"
#include "trepb_sys.h"
#include "trepb_varied.h"

namespace trepb {

struct CoopSys {
    int nl, nq, nd, nk, nu, nc, np, npairs, nlevels;
    int nsl;        // super levels of the pose sweep: one per run of single-child links (chain)
    int ndc, nqc;   // dynamic configs / configs that any constraint depends on (compact DDh.lambda block)
    int ns, nqs;    // LinearSpring potentials / configs that any of them depends on (compact block of their Hessian)
    int npc;        // points [0, npc) belong to constraints, [npc, np) are spring / damper ends (evaluated at the midpoint)
    int nfd, nqf;   // LinearDamper forces / configs that move exactly one end of any of them (compact f_dq, f_ddq blocks)
    int nns;        // NonlinearConfigSpring potentials (piecewise-quintic splines of one config)
    int nw;         // Body / Hybrid / Spatial wrench forces
    int has_gravity;
    double grav[3];
    // Tables live in one relocatable blob (host memory, device memory or a shared-memory copy):
    // `base` + byte offsets, so that moving the view is one pointer.
    //   links [nl]    l_par (parent link or -1), l_cfg (driving config), l_kind (bit0-1 axis, bit2
    //                 revolute, bit3 has pre-transform, bit4 carries mass below, bit5 carries a point
    //                 below), l_child0 / l_nchild (children are contiguous), l_Rc [nl][9], l_pc [nl][3],
    //                 l_in [nl][10] = m, h[3], Ibar (xx yy zz xy xz yz), l_anc (ancestor-or-self mask)
    //   lvl_off [nlevels+1]
    //   chains        l_next [nl] (the only child of a link, or -1), sl_off [nsl+1] / sl_head: the heads of
    //                 the chains (runs of single-child links) grouped by their depth in the tree of chains
    //   configs [nq]  cfg_link (link driven by the config or -1), damp [nd] (sum of Damping
    //                 coefficients), ks / kq0 [nq] (sum of ConfigSpring k, k*q0), Fu [nd][nu]
    //   pairs         pair_ij [npairs] = i | j << 8 (i ancestor-or-self of j); pm [nq][nd] = +idx+1 when
    //                 the row config is the ancestor(-or-self), -(idx+1) when it is the descendant, 0
    //   points [np]   pt_link (-1: fixed in the world), pt_r [np][3]
    //   constraints   con_kind, con_a, con_b (points), con_third, con_dist, con_tol, con_dep (config mask),
    //                 cd_off [nc+1] / cd_cfg: the configs each constraint depends on, ascending (the
    //                 first cd_nd[c] of them are dynamic); dd_row [nd] / dd_col [nq]: compact row / column
    //                 of a config in the block of sum_c lambda_c d2h_c (-1: no constraint depends on it);
    //                 con_n [nc][3]: PointOnPlane normal in the coordinates of the plane frame's link
    //   springs [ns]  LinearSpring (potentials/linearspring.c:30-74): sp_a, sp_b (points), sp_k, sp_x0,
    //                 sp_off [ns+1] / sp_cfg: the configs each spring depends on, ascending; xs_idx [nq]: compact
    //                 row = column of a config in the block of sum_s d2V_s / dq dq (-1: no spring depends on
    //                 it), xs_cfg [nqs] its inverse.  Links that carry a spring end have bit6 of l_kind set
    //                 (they take part in the midpoint pose sweep even without mass below).
    //   dampers [nfd] LinearDamper over a single-segment tape measure (forces/lineardamper.c:14-107,
    //                 tapemeasure.py:97-110): da_a, da_b (points), da_c, dp_off [nfd+1] / dp_cfg: the configs that
    //                 move exactly ONE end (the only ones the reference's path length depends on), xf_idx [nq] /
    //                 xf_cfg [nqf]: compact row = column of such a config in the f_dq / f_ddq blocks.
    //   spline springs [nns]  NonlinearConfigSpring (potentials/nonlinear_config_spring.c:23-47, spline.c:7-62):
    //                 nsp_i [nns][3] = config, offset into nsp_tab, number of x points; nsp_d [nns][2] = m, b;
    //                 nsp_tab: per spring x [n] then coefficients [n-1][6] (highest power first).
    //   wrenches [nw] forces/bodywrench.c, hybridwrench.c, spatialwrench.c: wr_i [nw][8] = kind, point, six input
    //                 indices (-1: constant component); wr_d [nw][15] = six constants, rotation of the frame in the
    //                 coordinates of its link (row-major 3x3); wr_dep [nw] config mask.  Their configs share the
    //                 compact f_dq block of the dampers (xf_idx / xf_cfg).
    const char* base;
    int o_l_par;
    int o_l_cfg;
    int o_l_kind;
    int o_l_child0;
    int o_l_nchild;
    int o_l_Rc;
    int o_l_pc;
    int o_l_in;
    int o_l_anc;
    int o_lvl_off;
    int o_cfg_link;
    int o_damp;
    int o_ks;
    int o_kq0;
    int o_Fu;
    int o_pair_ij;
    int o_pm;
    int o_pt_link;
    int o_pt_r;
    int o_con_kind;
    int o_con_a;
    int o_con_b;
    int o_con_third;
    int o_con_dist;
    int o_con_tol;
    int o_con_dep;
    int o_cd_off;
    int o_cd_cfg;
    int o_cd_nd;
    int o_dd_row;
    int o_dd_col;
    int o_l_next;
    int o_sl_off;
    int o_sl_head;
    int o_con_n;
    int o_sp_a, o_sp_b, o_sp_k, o_sp_x0, o_sp_off, o_sp_cfg, o_xs_idx, o_xs_cfg;
    int o_da_a, o_da_b, o_da_c, o_dp_off, o_dp_cfg, o_xf_idx, o_xf_cfg;
    int o_nsp_i, o_nsp_d, o_nsp_tab;
    int o_wr_i, o_wr_d, o_wr_dep;
    TREPB_HD const int32_t* wr_i() const { return (const int32_t*)(base + o_wr_i); }
    TREPB_HD const double* wr_d() const { return (const double*)(base + o_wr_d); }
    TREPB_HD const uint64_t* wr_dep() const { return (const uint64_t*)(base + o_wr_dep); }
    TREPB_HD const int32_t* nsp_i() const { return (const int32_t*)(base + o_nsp_i); }
    TREPB_HD const double* nsp_d() const { return (const double*)(base + o_nsp_d); }
    TREPB_HD const double* nsp_tab() const { return (const double*)(base + o_nsp_tab); }
    TREPB_HD const int32_t* da_a() const { return (const int32_t*)(base + o_da_a); }
    TREPB_HD const int32_t* da_b() const { return (const int32_t*)(base + o_da_b); }
    TREPB_HD const double* da_c() const { return (const double*)(base + o_da_c); }
    TREPB_HD const int32_t* dp_off() const { return (const int32_t*)(base + o_dp_off); }
    TREPB_HD const int32_t* dp_cfg() const { return (const int32_t*)(base + o_dp_cfg); }
    TREPB_HD const int32_t* xf_idx() const { return (const int32_t*)(base + o_xf_idx); }
    TREPB_HD const int32_t* xf_cfg() const { return (const int32_t*)(base + o_xf_cfg); }
    TREPB_HD const int32_t* sp_a() const { return (const int32_t*)(base + o_sp_a); }
    TREPB_HD const int32_t* sp_b() const { return (const int32_t*)(base + o_sp_b); }
    TREPB_HD const double* sp_k() const { return (const double*)(base + o_sp_k); }
    TREPB_HD const double* sp_x0() const { return (const double*)(base + o_sp_x0); }
    TREPB_HD const int32_t* sp_off() const { return (const int32_t*)(base + o_sp_off); }
    TREPB_HD const int32_t* sp_cfg() const { return (const int32_t*)(base + o_sp_cfg); }
    TREPB_HD const int32_t* xs_idx() const { return (const int32_t*)(base + o_xs_idx); }
    TREPB_HD const int32_t* xs_cfg() const { return (const int32_t*)(base + o_xs_cfg); }
    TREPB_HD const double* con_n() const { return (const double*)(base + o_con_n); }
    TREPB_HD const int32_t* l_par() const { return (const int32_t*)(base + o_l_par); }
    TREPB_HD const int32_t* l_cfg() const { return (const int32_t*)(base + o_l_cfg); }
    TREPB_HD const int32_t* l_kind() const { return (const int32_t*)(base + o_l_kind); }
    TREPB_HD const int32_t* l_child0() const { return (const int32_t*)(base + o_l_child0); }
    TREPB_HD const int32_t* l_nchild() const { return (const int32_t*)(base + o_l_nchild); }
    TREPB_HD const double* l_Rc() const { return (const double*)(base + o_l_Rc); }
    TREPB_HD const double* l_pc() const { return (const double*)(base + o_l_pc); }
    TREPB_HD const double* l_in() const { return (const double*)(base + o_l_in); }
    TREPB_HD const uint64_t* l_anc() const { return (const uint64_t*)(base + o_l_anc); }
    TREPB_HD const int32_t* lvl_off() const { return (const int32_t*)(base + o_lvl_off); }
    TREPB_HD const int32_t* cfg_link() const { return (const int32_t*)(base + o_cfg_link); }
    TREPB_HD const double* damp() const { return (const double*)(base + o_damp); }
    TREPB_HD const double* ks() const { return (const double*)(base + o_ks); }
    TREPB_HD const double* kq0() const { return (const double*)(base + o_kq0); }
    TREPB_HD const double* Fu() const { return (const double*)(base + o_Fu); }
    TREPB_HD const int32_t* pair_ij() const { return (const int32_t*)(base + o_pair_ij); }
    TREPB_HD const int16_t* pm() const { return (const int16_t*)(base + o_pm); }
    TREPB_HD const int32_t* pt_link() const { return (const int32_t*)(base + o_pt_link); }
    TREPB_HD const double* pt_r() const { return (const double*)(base + o_pt_r); }
    TREPB_HD const int32_t* con_kind() const { return (const int32_t*)(base + o_con_kind); }
    TREPB_HD const int32_t* con_a() const { return (const int32_t*)(base + o_con_a); }
    TREPB_HD const int32_t* con_b() const { return (const int32_t*)(base + o_con_b); }
    TREPB_HD const int32_t* con_third() const { return (const int32_t*)(base + o_con_third); }
    TREPB_HD const double* con_dist() const { return (const double*)(base + o_con_dist); }
    TREPB_HD const double* con_tol() const { return (const double*)(base + o_con_tol); }
    TREPB_HD const uint64_t* con_dep() const { return (const uint64_t*)(base + o_con_dep); }
    TREPB_HD const int32_t* cd_off() const { return (const int32_t*)(base + o_cd_off); }
    TREPB_HD const int32_t* cd_cfg() const { return (const int32_t*)(base + o_cd_cfg); }
    TREPB_HD const int32_t* cd_nd() const { return (const int32_t*)(base + o_cd_nd); }
    TREPB_HD const int32_t* dd_row() const { return (const int32_t*)(base + o_dd_row); }
    TREPB_HD const int32_t* dd_col() const { return (const int32_t*)(base + o_dd_col); }
    TREPB_HD const int32_t* l_next() const { return (const int32_t*)(base + o_l_next); }
    TREPB_HD const int32_t* sl_off() const { return (const int32_t*)(base + o_sl_off); }
    TREPB_HD const int32_t* sl_head() const { return (const int32_t*)(base + o_sl_head); }
    TREPB_HD int axis(int l) const { return l_kind()[l] & 3; }
    TREPB_HD bool rot(int l) const { return (l_kind()[l] & 4) != 0; }
    TREPB_HD bool has_xc(int l) const { return (l_kind()[l] & 8) != 0; }
    TREPB_HD bool dyn(int l) const { return (l_kind()[l] & 16) != 0; }
    TREPB_HD bool wrl(int l) const { return (l_kind()[l] & 32) != 0; }
};

// ---- the numeric part of the condensation
// coop_pack is a host-only PLAN - the topology, and which numbers of the description feed which numeric entry of the
// blob, in which order - followed by coop_eval_level / coop_eval_tables, which evaluate those entries from the plan
// and one numeric vector of the description: the table-driven kernels' expansion of a row (trepb_varied.h,
// slots = false: the numeric region of the packed blob, then grav[3]).  coop_pack runs them on the description's own
// vector; the varied cooperative kernels (TREPB_FLAG_COOP_VARIED) run them on a team's copy of the blob for the
// team's row.  The integer tables depend on structure only, which a varied entry never changes (varied_check).
//
// Every product and sum is rounded on its own, in the order the host evaluates it (x86-64 does not contract
// `a * b + c`; nvcc would, into an FMA), and every sum runs over its terms in ascending order, so the device gives
// the host's bits.  The one exception is cos / sin of a constant rotation frame's angle (K_RX .. K_RZ): the device
// math library and the C library may differ in the last bit.
TREPB_HD double cp_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
TREPB_HD double cp_add(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}

// The plan: sizes, indices and integer lists (one relocatable int32 array, like the blob).
struct CoopPlanView {
    int nlev;                            // depth levels of the frame tree
    int nl, np, nplane, nw, ncp, nsum;
    int xv, xs, xm, xg;                  // index in the numeric vector of frame_value[0], frame_se3[0], frame_mass[0], grav[0]
    int dRc, dpc, din, dpt, dcn, dwr;    // index (in doubles) in the blob of l_Rc, l_pc, l_in, pt_r, con_n, wr_d
    const int32_t* fr;       // [nf][3] every frame, level by level: frame, parent, kind (-1: identity - the world or a
                             // variable frame, whose link coordinates start at itself)
    const int32_t* fr_off;   // [nlev + 1]
    const int32_t* lk;       // [nl] the frame whose pose is link l's constant pre-transform (the parent of its frame)
    const int32_t* ms_off;   // [nl + 1] / ms: the frames whose masses sum into link l's inertia, ascending
    const int32_t* ms;
    const int32_t* pt;       // [np] frame of each point
    const int32_t* pl;       // [nplane][3] PointOnPlane constraint, plane frame, numeric index of its con_d[4 c]
    const int32_t* wr;       // [nw] frame of each wrench
    const int32_t* cp;       // [ncp][2] blob index <- numeric index
    const int32_t* sum_off;  // [nsum + 1], sum_dst [nsum], sum_t [][2]: blob index <- 0 + x[a] (b < 0) or x[a] * x[b] + ...
    const int32_t* sum_dst;
    const int32_t* sum_t;
};

// fx[12 f]: the pose of frame f in the coordinates of its link (of the world for a frame fixed in it), R row-major
// then p.  Level L of the frame tree; levels in order, each after the previous one is complete.
template <class X>
TREPB_HD void coop_eval_level(const CoopPlanView& pl, const X& x, double* fx, int L, int lane, int nlanes) {
    for (int i = pl.fr_off[L] + lane; i < pl.fr_off[L + 1]; i += nlanes) {
        const int f = pl.fr[3 * i], kind = pl.fr[3 * i + 2];
        double* o = fx + 12 * f;
        // local transform of a constant frame (trep/_trep/frame.c:839-1076)
        double b[12];
        for (int k = 0; k < 12; ++k) b[k] = (k < 9 && k % 4 == 0) ? 1.0 : 0.0;
        if (kind < 0) {
            for (int k = 0; k < 12; ++k) o[k] = b[k];
            continue;
        }
        if (kind == K_CONST_SE3) {
            for (int r = 0; r < 3; ++r) {
                for (int c = 0; c < 3; ++c) b[r * 3 + c] = x(pl.xs + 12 * f + r * 4 + c);
                b[9 + r] = x(pl.xs + 12 * f + r * 4 + 3);
            }
        } else if (kind >= K_TX && kind <= K_TZ) {
            b[9 + kind - K_TX] = x(pl.xv + f);
        } else if (kind >= K_RX && kind <= K_RZ) {
            const int a = kind - K_RX, bb = (a + 1) % 3, c = (a + 2) % 3;
            const double v = x(pl.xv + f), cs = cos(v), sn = sin(v);
            b[bb * 3 + bb] = cs; b[bb * 3 + c] = -sn;
            b[c * 3 + bb] = sn; b[c * 3 + c] = cs;
        }
        // parent then the local transform
        const double* a = fx + 12 * pl.fr[3 * i + 1];
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c)
                o[r * 3 + c] = cp_add(cp_add(cp_mul(a[r * 3], b[c]), cp_mul(a[r * 3 + 1], b[3 + c])), cp_mul(a[r * 3 + 2], b[6 + c]));
            o[9 + r] = cp_add(cp_add(cp_add(a[9 + r], cp_mul(a[r * 3], b[9])), cp_mul(a[r * 3 + 1], b[10])), cp_mul(a[r * 3 + 2], b[11]));
        }
    }
}

// Every numeric entry of the blob from the frame poses and the numeric vector; lanes split the destinations.
template <class X>
TREPB_HD void coop_eval_tables(const CoopPlanView& pl, const X& x, const double* fx, double* blob, int lane, int nlanes) {
    for (int l = lane; l < pl.nl; l += nlanes) {
        const double* xc = fx + 12 * pl.lk[l];
        for (int k = 0; k < 9; ++k) blob[pl.dRc + 9 * l + k] = xc[k];
        for (int k = 0; k < 3; ++k) blob[pl.dpc + 3 * l + k] = xc[9 + k];
        // masses -> link inertia (about the link origin, link axes): m, h = m c, R diag(Ixx, Iyy, Izz) R^T + m (|p|^2 1 - p p^T)
        double I[10];
        for (int k = 0; k < 10; ++k) I[k] = 0.0;
        for (int j = pl.ms_off[l]; j < pl.ms_off[l + 1]; ++j) {
            const int f = pl.ms[j];
            const double* R = fx + 12 * f;
            const double* p = R + 9;
            const double m = x(pl.xm + 4 * f);
            I[0] = cp_add(I[0], m);
            for (int k = 0; k < 3; ++k) I[1 + k] = cp_add(I[1 + k], cp_mul(m, p[k]));
            const double pp = cp_add(cp_add(cp_mul(p[0], p[0]), cp_mul(p[1], p[1])), cp_mul(p[2], p[2]));
            const int rr[6] = {0, 1, 2, 0, 0, 1}, cc[6] = {0, 1, 2, 1, 2, 2};
            for (int e = 0; e < 6; ++e) {
                const int r = rr[e], c = cc[e];
                double v = 0.0;
                for (int k = 0; k < 3; ++k) v = cp_add(v, cp_mul(cp_mul(R[r * 3 + k], x(pl.xm + 4 * f + 1 + k)), R[c * 3 + k]));
                v = cp_add(v, cp_mul(cp_mul(-m, p[r]), p[c]));
                if (r == c) v = cp_add(v, cp_mul(m, pp));
                I[4 + e] = cp_add(I[4 + e], v);
            }
        }
        for (int k = 0; k < 10; ++k) blob[pl.din + 10 * l + k] = I[k];
    }
    for (int i = lane; i < pl.np; i += nlanes)
        for (int k = 0; k < 3; ++k) blob[pl.dpt + 3 * i + k] = fx[12 * pl.pt[i] + 9 + k];
    // PointOnPlane: the normal, fixed in the plane frame, in the coordinates of the link the frame hangs on
    for (int i = lane; i < pl.nplane; i += nlanes) {
        const int c = pl.pl[3 * i], xn = pl.pl[3 * i + 2];
        const double* R = fx + 12 * pl.pl[3 * i + 1];
        const double n0 = x(xn), n1 = x(xn + 2), n2 = x(xn + 3);
        for (int r = 0; r < 3; ++r)
            blob[pl.dcn + 3 * c + r] = cp_add(cp_add(cp_mul(R[r * 3], n0), cp_mul(R[r * 3 + 1], n1)), cp_mul(R[r * 3 + 2], n2));
    }
    for (int i = lane; i < pl.nw; i += nlanes)
        for (int k = 0; k < 9; ++k) blob[pl.dwr + 15 * i + 6 + k] = fx[12 * pl.wr[i] + k];
    for (int i = lane; i < pl.ncp; i += nlanes) blob[pl.cp[2 * i]] = x(pl.cp[2 * i + 1]);
    for (int i = lane; i < pl.nsum; i += nlanes) {
        double v = 0.0;
        for (int j = pl.sum_off[i]; j < pl.sum_off[i + 1]; ++j) {
            const int a = pl.sum_t[2 * j], b = pl.sum_t[2 * j + 1];
            v = cp_add(v, b < 0 ? x(a) : cp_mul(x(a), x(b)));
        }
        blob[pl.sum_dst[i]] = v;
    }
}

// The numeric vector as an array (the host's).
struct CoopXVec {
    const double* v;
    TREPB_HD double operator()(int i) const { return v[i]; }
};

struct CoopPlan {
    std::vector<int32_t> ints;
    CoopPlanView hdr;    // sizes and indices; view() fills the pointers
    size_t o[12];        // offsets in ints of fr, fr_off, lk, ms_off, ms, pt, pl, wr, cp, sum_off, sum_dst, sum_t
    int nf = 0;          // frames (the frame poses take 12 nf doubles)
    CoopPlanView view(const int32_t* base) const {
        CoopPlanView v = hdr;
        const int32_t** p[12] = {&v.fr, &v.fr_off, &v.lk, &v.ms_off, &v.ms, &v.pt, &v.pl, &v.wr, &v.cp, &v.sum_off,
                                 &v.sum_dst, &v.sum_t};
        for (int k = 0; k < 12; ++k) *p[k] = base + o[k];
        return v;
    }
};

struct CoopPack {
    bool ok = false;
    std::string why;          // why the cooperative path does not apply
    std::vector<char> blob;
    CoopSys proto;
    size_t off[72];
    CoopPlan plan;           // evaluates the numeric tables of the blob from a numeric vector of the description

    CoopSys view(const char* base) const {
        CoopSys s = proto;
        s.base = base;
        int k = 0;
        s.o_l_par = (int)off[k++];
        s.o_l_cfg = (int)off[k++];
        s.o_l_kind = (int)off[k++];
        s.o_l_child0 = (int)off[k++];
        s.o_l_nchild = (int)off[k++];
        s.o_l_Rc = (int)off[k++];
        s.o_l_pc = (int)off[k++];
        s.o_l_in = (int)off[k++];
        s.o_l_anc = (int)off[k++];
        s.o_lvl_off = (int)off[k++];
        s.o_cfg_link = (int)off[k++];
        s.o_damp = (int)off[k++];
        s.o_ks = (int)off[k++];
        s.o_kq0 = (int)off[k++];
        s.o_Fu = (int)off[k++];
        s.o_pair_ij = (int)off[k++];
        s.o_pm = (int)off[k++];
        s.o_pt_link = (int)off[k++];
        s.o_pt_r = (int)off[k++];
        s.o_con_kind = (int)off[k++];
        s.o_con_a = (int)off[k++];
        s.o_con_b = (int)off[k++];
        s.o_con_third = (int)off[k++];
        s.o_con_dist = (int)off[k++];
        s.o_con_tol = (int)off[k++];
        s.o_con_dep = (int)off[k++];
        s.o_cd_off = (int)off[k++];
        s.o_cd_cfg = (int)off[k++];
        s.o_cd_nd = (int)off[k++];
        s.o_dd_row = (int)off[k++];
        s.o_dd_col = (int)off[k++];
        s.o_l_next = (int)off[k++];
        s.o_sl_off = (int)off[k++];
        s.o_sl_head = (int)off[k++];
        s.o_con_n = (int)off[k++];
        s.o_sp_a = (int)off[k++]; s.o_sp_b = (int)off[k++]; s.o_sp_k = (int)off[k++]; s.o_sp_x0 = (int)off[k++];
        s.o_sp_off = (int)off[k++]; s.o_sp_cfg = (int)off[k++]; s.o_xs_idx = (int)off[k++]; s.o_xs_cfg = (int)off[k++];
        s.o_da_a = (int)off[k++]; s.o_da_b = (int)off[k++]; s.o_da_c = (int)off[k++]; s.o_dp_off = (int)off[k++];
        s.o_dp_cfg = (int)off[k++]; s.o_xf_idx = (int)off[k++]; s.o_xf_cfg = (int)off[k++];
        s.o_nsp_i = (int)off[k++]; s.o_nsp_d = (int)off[k++]; s.o_nsp_tab = (int)off[k++];
        s.o_wr_i = (int)off[k++]; s.o_wr_d = (int)off[k++]; s.o_wr_dep = (int)off[k++];
        return s;
    }
};

// Builds the link-level tables.  Returns a pack with ok == false (and `why`) when the system uses
// something the cooperative kernels do not implement (the thread-per-instance general kernels do).
// P.plan evaluates the numeric tables for any numeric vector of the description (see above).
inline CoopPack coop_pack(const trepb_sysdesc* d) {
    CoopPack P;
    const int nf = d->n_frames, nd = d->nd, nk = d->nk, nq = nd + nk, nu = d->nu, nc = d->n_constraints;
    if (nq > 64) { P.why = "more than 64 configs"; return P; }
    for (int i = 0; i < d->n_forces; ++i)
        if (d->force_kind[i] == TREPB_FORCE_LINEAR_DAMPER && d->force_i[4 * i + 1] != 2) { P.why = "LinearDamper over more than one segment"; return P; }
    // the description's numeric vector, laid out as the expansion of a row lays it out
    std::vector<double> xv;
    int toff[8];
    {
        PackedSys PS;
        std::string err;
        if (!pack_system(d, &PS, &err)) { P.why = err; return P; }
        VariedHost H;
        varied_map(PS, 0, nullptr, nullptr, false, &H);
        xv = H.base;
        for (int k = 0; k < 8; ++k) toff[k] = H.toff[k];
    }
    const CoopXVec X{xv.data()};
    CoopPlan& PL = P.plan;
    PL.nf = nf;
    CoopPlanView& hd = PL.hdr;
    memset(&hd, 0, sizeof(hd));
    hd.xv = toff[0]; hd.xs = toff[1]; hd.xm = toff[2]; hd.xg = toff[7];

    // ---- frames -> links
    std::vector<int> flink(nf, -1);      // frame -> frame index of the link it belongs to (-1: world)
    std::vector<int> lframes;            // variable frames in pre-order
    std::vector<int> fdepth(nf, 0);
    int nfl = 1;
    for (int f = 1; f < nf; ++f) {
        const int par = d->frame_parent[f];
        fdepth[f] = fdepth[par] + 1;
        if (fdepth[f] + 1 > nfl) nfl = fdepth[f] + 1;
        if (d->frame_config[f] >= 0) {
            flink[f] = f;
            lframes.push_back(f);
        } else {
            flink[f] = flink[par];
        }
    }
    // frame poses in their links' coordinates, level by level of the frame tree
    std::vector<int32_t> fr, fr_off;
    for (int L = 0; L < nfl; ++L) {
        fr_off.push_back((int32_t)(fr.size() / 3));
        for (int f = 0; f < nf; ++f) {
            if (fdepth[f] != L) continue;
            fr.push_back(f);
            fr.push_back(f == 0 ? 0 : d->frame_parent[f]);
            fr.push_back(f == 0 || d->frame_config[f] >= 0 ? -1 : d->frame_kind[f]);
        }
    }
    fr_off.push_back((int32_t)(fr.size() / 3));
    hd.nlev = nfl;
    std::vector<double> fxv((size_t)12 * nf);
    {
        CoopPlanView fv = hd;
        fv.fr = fr.data(); fv.fr_off = fr_off.data();
        for (int L = 0; L < nfl; ++L) coop_eval_level(fv, X, fxv.data(), L, 0, 1);
    }
    auto fx_identity = [&](int f) {
        const double* x = &fxv[(size_t)12 * f];
        for (int k = 0; k < 9; ++k) if (x[k] != ((k % 4 == 0) ? 1.0 : 0.0)) return false;
        return x[9] == 0.0 && x[10] == 0.0 && x[11] == 0.0;
    };
    const int nl = (int)lframes.size();
    if (nl < 1) { P.why = "no variable frame"; return P; }
    if (nl > 64) { P.why = "more than 64 variable frames"; return P; }
    // parent link (as frame index) and level of every variable frame
    std::vector<int> fpl(nf, -1), flevel(nf, 0);
    int nlevels = 0;
    for (int f : lframes) {
        fpl[f] = flink[d->frame_parent[f]];
        flevel[f] = fpl[f] < 0 ? 0 : flevel[fpl[f]] + 1;
        if (flevel[f] + 1 > nlevels) nlevels = flevel[f] + 1;
    }
    // level order; within a level, ordered by (parent's new index, pre-order) so children are contiguous
    std::vector<int> order;              // new link index -> frame
    std::vector<int> newidx(nf, -1);
    std::vector<int32_t> lvl_off(nlevels + 1, 0);
    for (int L = 0; L < nlevels; ++L) {
        lvl_off[L] = (int32_t)order.size();
        if (L == 0) {
            for (int f : lframes) if (flevel[f] == 0) { newidx[f] = (int)order.size(); order.push_back(f); }
        } else {
            const int lo = lvl_off[L - 1], hi = (int)order.size();
            for (int pi = lo; pi < hi; ++pi)
                for (int f : lframes)
                    if (flevel[f] == L && fpl[f] == order[pi]) { newidx[f] = (int)order.size(); order.push_back(f); }
        }
    }
    lvl_off[nlevels] = (int32_t)order.size();

    // numeric entries: (table of the blob in put order, element) <- one numeric-vector entry, or a sum of terms
    struct Dst { int tab, pos; };
    std::vector<std::pair<Dst, int>> copies;
    std::vector<std::pair<Dst, std::vector<std::pair<int, int>>>> sums;
    enum { T_DAMP = 11, T_KS = 12, T_KQ0 = 13, T_CON_DIST = 23, T_CON_TOL = 24, T_SP_K = 37, T_SP_X0 = 38, T_DA_C = 45,
           T_NSP_D = 51, T_NSP_TAB = 52, T_WR_D = 54 };
    const int xpot = toff[3], xforce = toff[4], xcon = toff[5], xpool = toff[6];

    std::vector<int32_t> l_par(nl), l_cfg(nl), l_kind(nl), l_child0(nl, 0), l_nchild(nl, 0);
    std::vector<double> l_Rc(9 * nl, 0.0), l_pc(3 * nl, 0.0), l_in(10 * nl, 0.0);
    std::vector<uint64_t> l_anc(nl, 0);
    std::vector<int32_t> cfg_link(nq > 0 ? nq : 1, -1), lk(nl);
    for (int l = 0; l < nl; ++l) {
        const int f = order[l];
        const int kind = d->frame_kind[f];
        l_par[l] = fpl[f] < 0 ? -1 : newidx[fpl[f]];
        l_cfg[l] = d->frame_config[f];
        cfg_link[l_cfg[l]] = l;
        lk[l] = d->frame_parent[f];
        int kbits = (kind >= K_RX ? (kind - K_RX) | 4 : (kind - K_TX));
        if (!fx_identity(lk[l])) kbits |= 8;
        l_kind[l] = kbits;
        l_anc[l] = (l_par[l] < 0 ? 0ull : l_anc[l_par[l]]) | (1ull << l);
    }
    for (int l = nl - 1; l >= 0; --l)
        if (l_par[l] >= 0) { l_child0[l_par[l]] = l; l_nchild[l_par[l]]++; }

    // ---- chains: a lane of the pose sweep follows a run of single-child links without going through
    // shared memory; the heads of the chains are grouped by their depth in the tree of chains
    std::vector<int32_t> l_next(nl, -1), sl_off, sl_head;
    int nsl = 0;
    {
        for (int l = 0; l < nl; ++l) if (l_nchild[l] == 1) l_next[l] = l_child0[l];
        std::vector<int> cdepth(nl, 0);
        std::vector<std::vector<int32_t>> by_depth;
        for (int l = 0; l < nl; ++l) {
            const int par = l_par[l];
            const bool head = par < 0 || l_nchild[par] != 1;
            cdepth[l] = par < 0 ? 0 : cdepth[par] + (head ? 1 : 0);
            if (head) {
                if ((int)by_depth.size() <= cdepth[l]) by_depth.resize(cdepth[l] + 1);
                by_depth[cdepth[l]].push_back(l);
            }
        }
        nsl = (int)by_depth.size();
        for (int dth = 0; dth < nsl; ++dth) {
            sl_off.push_back((int32_t)sl_head.size());
            for (int32_t l : by_depth[dth]) sl_head.push_back(l);
        }
        sl_off.push_back((int32_t)sl_head.size());
    }

    // ---- masses -> link inertia: which frames, in ascending order
    std::vector<std::vector<int32_t>> lmass(nl);
    for (int f = 1; f < nf; ++f) {
        const double* mm = d->frame_mass + 4 * f;
        if (mm[0] == 0.0 && mm[1] == 0.0 && mm[2] == 0.0 && mm[3] == 0.0) continue;
        if (flink[f] < 0) continue;  // fixed in the world: contributes nothing to the dynamics
        const int l = newidx[flink[f]];
        lmass[l].push_back(f);
        for (int a = l; a >= 0; a = l_par[a]) l_kind[a] |= 16;
    }

    // ---- constraint end points
    std::vector<int32_t> pt_link;
    std::vector<double> pt_r;
    std::vector<int> pt_frame;
    // first: search from this point index (spring ends get their own points even when a constraint uses the
    // same frame: the two sets are evaluated at different poses); bit: the l_kind flag of the links above it
    auto point_of = [&](int f, size_t first = 0, int bit = 32) {
        for (size_t i = first; i < pt_frame.size(); ++i) if (pt_frame[i] == f) return (int)i;
        pt_frame.push_back(f);
        const int l = flink[f] < 0 ? -1 : newidx[flink[f]];
        pt_link.push_back(l);
        for (int k = 0; k < 3; ++k) pt_r.push_back(0.0);
        for (int a = l; a >= 0; a = l_par[a]) l_kind[a] |= bit;
        return (int)pt_frame.size() - 1;
    };
    std::vector<int32_t> con_kind(nc > 0 ? nc : 1), con_a(nc > 0 ? nc : 1), con_b(nc > 0 ? nc : 1), con_third(nc > 0 ? nc : 1);
    std::vector<double> con_dist(nc > 0 ? nc : 1, 0.0), con_tol(nc > 0 ? nc : 1, 0.0);
    std::vector<uint64_t> con_dep(nc > 0 ? nc : 1, 0);
    std::vector<double> con_n(nc > 0 ? 3 * nc : 3, 0.0);
    std::vector<int32_t> planes;
    for (int c = 0; c < nc; ++c) {
        const int32_t* ii = d->con_i + 4 * c;
        con_kind[c] = d->con_kind[c];
        con_a[c] = point_of(ii[0]);
        con_b[c] = point_of(ii[1]);
        con_third[c] = ii[2];
        copies.push_back({{T_CON_TOL, c}, xcon + 4 * c + 1});
        if (con_kind[c] == TREPB_CON_PLANE) {
            // normal (con_d[0], con_d[2], con_d[3]) fixed in the plane frame; distance 0
            planes.push_back(c); planes.push_back(ii[0]); planes.push_back(xcon + 4 * c);
            con_third[c] = -1;
        } else {
            copies.push_back({{T_CON_DIST, c}, xcon + 4 * c});
        }
        uint64_t m = 0;
        for (int e = 0; e < 2; ++e) {
            const int l = pt_link[e == 0 ? con_a[c] : con_b[c]];
            if (l < 0) continue;
            for (int a = l; a >= 0; a = l_par[a]) m |= 1ull << l_cfg[a];
        }
        if (con_kind[c] == TREPB_CON_DISTANCE && ii[2] >= 0) m |= 1ull << ii[2];
        con_dep[c] = m;
    }
    const int npc = (int)pt_link.size();
    // ---- LinearSpring end points and dependency lists
    std::vector<int32_t> sp_a, sp_b, sp_off(1, 0), sp_cfg;
    std::vector<double> sp_k, sp_x0;
    std::vector<int32_t> xs_idx(nq > 0 ? nq : 1, -1), xs_cfg;
    {
        uint64_t any = 0;
        for (int i = 0; i < d->n_potentials; ++i) {
            if (d->pot_kind[i] != TREPB_POT_LINEAR_SPRING) continue;
            const int a = point_of(d->pot_i[4 * i], (size_t)npc, 64), b = point_of(d->pot_i[4 * i + 1], (size_t)npc, 64);
            copies.push_back({{T_SP_K, (int)sp_a.size()}, xpot + 4 * i});
            copies.push_back({{T_SP_X0, (int)sp_a.size()}, xpot + 4 * i + 1});
            sp_a.push_back(a); sp_b.push_back(b);
            sp_k.push_back(0.0); sp_x0.push_back(0.0);
            uint64_t m = 0;
            for (int e = 0; e < 2; ++e) {
                const int l = pt_link[e == 0 ? a : b];
                for (int x = l; x >= 0; x = l_par[x]) m |= 1ull << l_cfg[x];
            }
            for (int j = 0; j < nq; ++j) if ((m >> j) & 1ull) sp_cfg.push_back(j);
            sp_off.push_back((int32_t)sp_cfg.size());
            any |= m;
        }
        for (int j = 0; j < nq; ++j) if ((any >> j) & 1ull) { xs_idx[j] = (int32_t)xs_cfg.size(); xs_cfg.push_back(j); }
    }
    const int ns = (int)sp_a.size(), nqs = (int)xs_cfg.size();
    // ---- LinearDamper end points and the configs that move exactly one end
    std::vector<int32_t> da_a, da_b, dp_off(1, 0), dp_cfg, xf_idx(nq > 0 ? nq : 1, -1), xf_cfg;
    std::vector<double> da_c, wr_d;
    std::vector<int32_t> wr_i, wr_frame;
    std::vector<uint64_t> wr_dep;
    {
        uint64_t any = 0;
        for (int i = 0; i < d->n_forces; ++i) {
            if (d->force_kind[i] != TREPB_FORCE_LINEAR_DAMPER) continue;
            const int off = d->force_i[4 * i];
            const int a = point_of(d->ipool[off], (size_t)npc, 64), b = point_of(d->ipool[off + 1], (size_t)npc, 64);
            copies.push_back({{T_DA_C, (int)da_a.size()}, xforce + 4 * i});
            da_a.push_back(a); da_b.push_back(b); da_c.push_back(0.0);
            uint64_t ma = 0, mb = 0;
            for (int x = pt_link[a]; x >= 0; x = l_par[x]) ma |= 1ull << l_cfg[x];
            for (int x = pt_link[b]; x >= 0; x = l_par[x]) mb |= 1ull << l_cfg[x];
            const uint64_t m = ma ^ mb;
            for (int j = 0; j < nq; ++j) if ((m >> j) & 1ull) dp_cfg.push_back(j);
            dp_off.push_back((int32_t)dp_cfg.size());
            any |= m;
        }
        for (int i = 0; i < d->n_forces; ++i) {
            const int kind = d->force_kind[i];
            if (kind < TREPB_FORCE_BODY_WRENCH) continue;
            const int f = d->force_i[4 * i], io = d->force_i[4 * i + 1], dof = d->force_i[4 * i + 2];
            const int pt = point_of(f, (size_t)npc, 64);
            wr_i.push_back(kind); wr_i.push_back(pt);
            for (int k = 0; k < 6; ++k) wr_i.push_back(d->ipool[io + k]);
            for (int k = 0; k < 6; ++k) copies.push_back({{T_WR_D, (int)wr_d.size() + k}, xpool + dof + k});
            for (int k = 0; k < 15; ++k) wr_d.push_back(0.0);
            wr_frame.push_back(f);
            uint64_t m = 0;
            for (int x = pt_link[pt]; x >= 0; x = l_par[x]) m |= 1ull << l_cfg[x];
            wr_dep.push_back(m);
            any |= m;
        }
        for (int j = 0; j < nq; ++j) if ((any >> j) & 1ull) { xf_idx[j] = (int32_t)xf_cfg.size(); xf_cfg.push_back(j); }
    }
    const int nfd = (int)da_a.size(), nqf = (int)xf_cfg.size(), nw = (int)wr_dep.size();
    // ---- NonlinearConfigSpring tables
    std::vector<int32_t> nsp_i;
    std::vector<double> nsp_d, nsp_tab;
    for (int i = 0; i < d->n_potentials; ++i) {
        if (d->pot_kind[i] != TREPB_POT_NONLINEAR_CONFIG_SPRING) continue;
        const int c = d->pot_i[4 * i], off = d->pot_i[4 * i + 1], n = d->pot_i[4 * i + 2];
        nsp_i.push_back(c); nsp_i.push_back((int32_t)nsp_tab.size()); nsp_i.push_back(n);
        copies.push_back({{T_NSP_D, (int)nsp_d.size()}, xpot + 4 * i});
        copies.push_back({{T_NSP_D, (int)nsp_d.size() + 1}, xpot + 4 * i + 1});
        nsp_d.push_back(0.0); nsp_d.push_back(0.0);
        for (int e = 0; e < n + 6 * (n - 1); ++e) {
            copies.push_back({{T_NSP_TAB, (int)nsp_tab.size()}, xpool + off + e});
            nsp_tab.push_back(0.0);
        }
    }
    const int nns = (int)nsp_i.size() / 3;
    const int np = (int)pt_link.size();
    std::vector<int32_t> cd_off(nc + 1, 0), cd_cfg, cd_nd(nc > 0 ? nc : 1, 0);
    for (int c = 0; c < nc; ++c) {
        cd_off[c] = (int32_t)cd_cfg.size();
        for (int j = 0; j < nq; ++j)
            if ((con_dep[c] >> j) & 1ull) { cd_cfg.push_back(j); if (j < nd) cd_nd[c]++; }
    }
    cd_off[nc] = (int32_t)cd_cfg.size();
    std::vector<int32_t> dd_row(nd > 0 ? nd : 1, -1), dd_col(nq > 0 ? nq : 1, -1);
    int ndc = 0, nqc = 0;
    {
        uint64_t any = 0;
        for (int c = 0; c < nc; ++c) any |= con_dep[c];
        for (int j = 0; j < nq; ++j)
            if ((any >> j) & 1ull) { dd_col[j] = nqc++; if (j < nd) dd_row[j] = ndc++; }
    }

    // ---- chain pairs (only links that carry mass below)
    std::vector<int32_t> pair_ij;
    std::vector<int16_t> pm((size_t)(nq * nd > 0 ? nq * nd : 1), 0);   // [nq][nd]: the column config is always dynamic
    for (int j = 0; j < nl; ++j) {
        if (!(l_kind[j] & 16)) continue;
        for (int i = j; i >= 0; i = l_par[i]) {
            const int idx = (int)pair_ij.size();
            pair_ij.push_back(i | (j << 8));
            const int ci = l_cfg[i], cj = l_cfg[j];
            if (cj < nd) pm[(size_t)ci * nd + cj] = (int16_t)(idx + 1);
            if (i != j && ci < nd) pm[(size_t)cj * nd + ci] = (int16_t)(-(idx + 1));
        }
    }
    const int npairs = (int)pair_ij.size();
    if (npairs > 30000) { P.why = "too many chain pairs"; return P; }

    // ---- potentials / forces folded into per-config constants: sums in potential / force order
    std::vector<double> damp(nd > 0 ? nd : 1, 0.0), ks(nq > 0 ? nq : 1, 0.0), kq0(nq > 0 ? nq : 1, 0.0), Fu((size_t)(nd * nu > 0 ? nd * nu : 1), 0.0);
    std::vector<std::vector<std::pair<int, int>>> t_damp(nd > 0 ? nd : 1), t_ks(nq > 0 ? nq : 1), t_kq0(nq > 0 ? nq : 1);
    int has_grav = 0;
    for (int i = 0; i < d->n_potentials; ++i) {
        if (d->pot_kind[i] == TREPB_POT_GRAVITY) {
            has_grav = 1;
        } else if (d->pot_kind[i] == TREPB_POT_CONFIG_SPRING) {
            const int c = d->pot_i[4 * i];
            t_ks[c].push_back({xpot + 4 * i, -1});
            t_kq0[c].push_back({xpot + 4 * i, xpot + 4 * i + 1});
        }
    }
    for (int i = 0; i < d->n_forces; ++i) {
        if (d->force_kind[i] == TREPB_FORCE_DAMPING) {
            for (int j = 0; j < nd; ++j) t_damp[j].push_back({xpool + d->force_i[4 * i] + j, -1});
        } else if (d->force_kind[i] == TREPB_FORCE_CONFIG) {
            const int c = d->force_i[4 * i], u = d->force_i[4 * i + 1];
            if (c < nd) Fu[(size_t)c * nu + u] += 1.0;
        }
    }
    for (int j = 0; j < nd; ++j) if (!t_damp[j].empty()) sums.push_back({{T_DAMP, j}, t_damp[j]});
    for (int j = 0; j < nq; ++j) if (!t_ks[j].empty()) sums.push_back({{T_KS, j}, t_ks[j]});
    for (int j = 0; j < nq; ++j) if (!t_kq0[j].empty()) sums.push_back({{T_KQ0, j}, t_kq0[j]});

    // ---- pack
    memset(&P.proto, 0, sizeof(P.proto));
    P.proto.nl = nl; P.proto.nq = nq; P.proto.nd = nd; P.proto.nk = nk; P.proto.nu = nu; P.proto.nc = nc;
    P.proto.np = np; P.proto.npairs = npairs; P.proto.nlevels = nlevels;
    P.proto.ndc = ndc; P.proto.nqc = nqc; P.proto.nsl = nsl;
    P.proto.ns = ns; P.proto.nqs = nqs; P.proto.npc = npc;
    P.proto.nfd = nfd; P.proto.nqf = nqf; P.proto.nns = nns; P.proto.nw = nw;
    P.proto.has_gravity = has_grav;
    for (int k = 0; k < 3; ++k) P.proto.grav[k] = X(hd.xg + k);
    int k = 0;
    auto put = [&](const void* src, size_t bytes) {
        size_t o = (P.blob.size() + 15) & ~size_t(15);
        P.blob.resize(o + (bytes ? bytes : 16), 0);
        if (bytes && src) memcpy(P.blob.data() + o, src, bytes);
        P.off[k++] = o;
    };
    put(l_par.data(), 4 * nl); put(l_cfg.data(), 4 * nl); put(l_kind.data(), 4 * nl);
    put(l_child0.data(), 4 * nl); put(l_nchild.data(), 4 * nl);
    put(l_Rc.data(), 8 * 9 * nl); put(l_pc.data(), 8 * 3 * nl); put(l_in.data(), 8 * 10 * nl);
    put(l_anc.data(), 8 * nl); put(lvl_off.data(), 4 * (nlevels + 1));
    put(cfg_link.data(), 4 * nq); put(damp.data(), 8 * nd); put(ks.data(), 8 * nq); put(kq0.data(), 8 * nq);
    put(Fu.data(), 8 * (size_t)nd * nu);
    put(pair_ij.data(), 4 * (size_t)npairs); put(pm.data(), 2 * (size_t)nq * nd);
    put(pt_link.data(), 4 * (size_t)np); put(pt_r.data(), 8 * 3 * (size_t)np);
    put(con_kind.data(), 4 * nc); put(con_a.data(), 4 * nc); put(con_b.data(), 4 * nc); put(con_third.data(), 4 * nc);
    put(con_dist.data(), 8 * nc); put(con_tol.data(), 8 * nc); put(con_dep.data(), 8 * nc);
    put(cd_off.data(), 4 * (nc + 1)); put(cd_cfg.data(), 4 * cd_cfg.size()); put(cd_nd.data(), 4 * nc);
    put(dd_row.data(), 4 * nd); put(dd_col.data(), 4 * nq);
    put(l_next.data(), 4 * nl); put(sl_off.data(), 4 * sl_off.size()); put(sl_head.data(), 4 * sl_head.size());
    put(con_n.data(), 8 * 3 * (size_t)nc);
    put(sp_a.data(), 4 * (size_t)ns); put(sp_b.data(), 4 * (size_t)ns); put(sp_k.data(), 8 * (size_t)ns); put(sp_x0.data(), 8 * (size_t)ns);
    put(sp_off.data(), 4 * sp_off.size()); put(sp_cfg.data(), 4 * sp_cfg.size());
    put(xs_idx.data(), 4 * (size_t)nq); put(xs_cfg.data(), 4 * (size_t)nqs);
    put(da_a.data(), 4 * (size_t)nfd); put(da_b.data(), 4 * (size_t)nfd); put(da_c.data(), 8 * (size_t)nfd);
    put(dp_off.data(), 4 * dp_off.size()); put(dp_cfg.data(), 4 * dp_cfg.size());
    put(xf_idx.data(), 4 * (size_t)nq); put(xf_cfg.data(), 4 * (size_t)nqf);
    put(nsp_i.data(), 4 * nsp_i.size()); put(nsp_d.data(), 8 * nsp_d.size()); put(nsp_tab.data(), 8 * nsp_tab.size());
    put(wr_i.data(), 4 * wr_i.size()); put(wr_d.data(), 8 * wr_d.size()); put(wr_dep.data(), 8 * wr_dep.size());
    P.blob.resize((P.blob.size() + 15) & ~size_t(15), 0);

    // ---- the plan, with blob positions resolved
    auto dst = [&](const Dst& t) { return (int32_t)(P.off[t.tab] / sizeof(double)) + t.pos; };
    hd.nl = nl; hd.np = np; hd.nplane = (int)planes.size() / 3; hd.nw = nw;
    hd.ncp = (int)copies.size(); hd.nsum = (int)sums.size();
    hd.dRc = (int)(P.off[5] / 8); hd.dpc = (int)(P.off[6] / 8); hd.din = (int)(P.off[7] / 8);
    hd.dpt = (int)(P.off[18] / 8); hd.dcn = (int)(P.off[34] / 8); hd.dwr = (int)(P.off[54] / 8);
    std::vector<int32_t>& I = PL.ints;
    I.clear();
    int ko = 0;
    auto add = [&](const std::vector<int32_t>& v) { PL.o[ko++] = I.size(); I.insert(I.end(), v.begin(), v.end()); };
    std::vector<int32_t> ms_off(1, 0), ms, pts(pt_frame.begin(), pt_frame.end()), cps, sum_off(1, 0), sum_dst, sum_t;
    for (int l = 0; l < nl; ++l) { ms.insert(ms.end(), lmass[l].begin(), lmass[l].end()); ms_off.push_back((int32_t)ms.size()); }
    for (const auto& c : copies) { cps.push_back(dst(c.first)); cps.push_back(c.second); }
    for (const auto& s : sums) {
        sum_dst.push_back(dst(s.first));
        for (const auto& t : s.second) { sum_t.push_back(t.first); sum_t.push_back(t.second); }
        sum_off.push_back((int32_t)(sum_t.size() / 2));
    }
    add(fr); add(fr_off); add(lk); add(ms_off); add(ms); add(pts); add(planes); add(wr_frame); add(cps); add(sum_off);
    add(sum_dst); add(sum_t);
    I.push_back(0);   // keeps every offset inside the array
    // ---- the numeric tables of the description
    coop_eval_tables(PL.view(I.data()), X, fxv.data(), (double*)P.blob.data(), 0, 1);
    P.ok = true;
    return P;
}

}  // namespace trepb
