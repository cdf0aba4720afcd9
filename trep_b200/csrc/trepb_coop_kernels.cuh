// Team-cooperative kernel templates: one TEAM (one warp, or two for the linearize kernel of shapes built with
// PairTeam) per instance, the per-instance workspace and the link tables in shared memory
// (trepb_coop_math.cuh).  Used for systems whose thread-per-instance workspace would not stay on chip (the
// marionette: 86 frames, nd 22, nk 18, nc 6).
//
//   coop_step_kernel     trepb_step_batch*       (MidpointVI.step looped in-kernel)
//   coop_project_kernel  trepb_project_batch*    (closed-loop rollouts)
//   coop_p2_kernel       trepb_calc_p2_batch* / trepb_calc_f_batch* / trepb_discrete_fm2_batch*
//   coop_lin_kernel      trepb_linearize_batch*  (solve_DEL + calc_deriv1 -> A, B, raw arrays, aux)
//
// Persistent grid: one CTA per SM, as many teams per CTA as workspaces fit next to the table blob in the SM's
// shared memory (marionette: 8 x 26.6 KB for the linearize kernel, 12 x 18.0 KB for the kernels that never
// call deriv1, + 12.3 KB of tables); every team walks the batch with stride grid x teams.  Cross-lane traffic
// goes through shared memory and the team's barrier (__syncwarp / a named barrier); the factorizations run on
// the team's first warp with shuffles and warp reductions.
#pragma once
#include <cuda_runtime.h>
#include "trepb_coop.h"

namespace trepb {
namespace coopk {

// CTA-wide barrier at the start of every instance / step (see coop_lin_kernel); -DTREPB_COOP_FREERUN
// lets the teams run free (experiment)
#if defined(TREPB_COOP_FREERUN)
#define TREPB_LOCKSTEP() ((void)0)
#else
#define TREPB_LOCKSTEP() __syncthreads()
#endif


struct Stage {
    CoopSys S;
    double* w;
};

// The team's index in its CTA as a value the compiler knows to be the same in all lanes of a warp (the
// result of a broadcast): the workspace base, the instance index and every branch taken on data read
// from the workspace are then provably warp-uniform, which removes the re-convergence bookkeeping (BSSY /
// BSYNC, WARPSYNC.COLLECTIVE around every shuffle and reduction) the compiler otherwise emits.
template <class Team>
__device__ __forceinline__ int team_index() {
    return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0) / Team::kWarps;
}
template <class Team>
__device__ __forceinline__ Team make_team() {
    if constexpr (Team::kWarps > 1) {
        Team t;
        t.bar = 1 + team_index<Team>();
        return t;
    } else {
        return Team();
    }
}

// layout of a compile-time-size flavour: constants from the template dimensions, plus - for CtDims<..., 1> - the
// run-time tail of the plugin kinds only some systems have (the same function the host sized the workspace with)
template <class D>
__device__ __forceinline__ CoopLayout static_layout(const CoopSys& gs, bool solve_only) {
    CoopLayout lay = D::layout(solve_only);
    if constexpr (D::kExtras) lay.append_extras(D::ND, D::ND + D::NK, D::NU, gs.nqs, gs.nqf, gs.nns, gs.nw);
    return lay;
}

// D::kExt / D::kExtS: this team's slab of the external region (one per team of the persistent grid)
template <class D, class Team>
__device__ __forceinline__ double* team_slab(double* ext, const CoopLayout& lay) {
    if constexpr (D::kExt || D::kExtS)
        return ext + ((long)blockIdx.x * (blockDim.x / Team::kSize) + team_index<Team>()) * lay.xtotal;
    else
        return nullptr;
}

template <class Team>
__device__ __forceinline__ Stage coop_stage(const CoopSys& gs, int blob_bytes, const CoopLayout& lay) {
    extern __shared__ double smem_[];
    const int n8 = (blob_bytes + 7) / 8;
    const double* src = (const double*)gs.base;
    for (int i = threadIdx.x; i < n8; i += blockDim.x) smem_[i] = src[i];
    __syncthreads();
    Stage st;
    st.S = gs;
    st.S.base = (const char*)smem_;
    st.w = smem_ + ((n8 + 1) & ~1) + (long)team_index<Team>() * lay.total;
    return st;
}

// Varied flavours (CoopVaried): the team's copy of the blob in its slot of scratch, the team's view of the system
// (grav: its row's) and the row whose numbers the copy holds.  The integer tables are copied once per launch, the
// numeric ones re-evaluated only when the team's row changes.
struct TeamTables {
    CoopSys S;
    double* fx;
    long row;
};

template <class Team>
__device__ __forceinline__ void varied_init(TeamTables& tt, const Stage& st, int blob_bytes, const CoopVaried& v, const Team& tm) {
    const long g = (long)blockIdx.x * (blockDim.x / Team::kSize) + team_index<Team>();
    double* slot = v.scratch + g * v.per_team;
    const int n8 = (blob_bytes + 7) / 8;
    const double* src = (const double*)st.S.base;
    for (int i = tm.lane(); i < n8; i += Team::kSize) slot[i] = src[i];
    tt.S = st.S;
    tt.S.base = (const char*)slot;
    tt.fx = slot + ((n8 + 1) & ~1);
    tt.row = -1;
}

// Points the team's tables at row r (the whole team calls it; the barriers order the slot's writes and reads).
template <class Team>
__device__ __forceinline__ void varied_row(TeamTables& tt, const CoopVaried& v, long r, const Team& tm) {
    if (r == tt.row) return;
    tm.sync();
    const VariedX x{v.map, v.values + r * v.map.n};
    for (int L = 0; L < v.plan.nlev; ++L) {
        coop_eval_level(v.plan, x, tt.fx, L, tm.lane(), Team::kSize);
        tm.sync();
    }
    coop_eval_tables(v.plan, x, tt.fx, (double*)tt.S.base, tm.lane(), Team::kSize);
    for (int k = 0; k < 3; ++k) tt.S.grav[k] = x(v.plan.xg + k);
    tt.row = r;
    tm.sync();
}

template <bool kVaried>
__device__ __forceinline__ const CoopSys& team_sys(const Stage& st, const TeamTables& tt) {
    if constexpr (kVaried) return tt.S;
    else return st.S;
}

template <class D, class Team, int TEAMS, bool kVaried>
__device__ __forceinline__ void
coop_step_body(const CoopSys& gs, const int blob_bytes, const CoopLayout& lay_, const StepParams& p, double* __restrict__ ext,
               const CoopVaried* v) {
    CoopLayout lay = lay_;
    if constexpr (D::kStatic) lay = static_layout<D>(gs, true);
    Stage st = coop_stage<Team>(gs, blob_bytes, lay);
    const Team tm = make_team<Team>();
    TeamTables tt;
    if constexpr (kVaried) varied_init(tt, st, blob_bytes, *v, tm);
    const CoopSys& S = team_sys<kVaried>(st, tt);
    double* w = st.w;
    constexpr int TS = Team::kSize;
    Coop<Team, D> c(S, lay, w, tm, team_slab<D, Team>(ext, lay));
    const int lane = tm.lane(), wpc = blockDim.x / TS;
    const int nd = c.ND(), nk = c.NK(), nq = c.NQ(), nu = c.NU(), nc = c.NC();
    // the warps of a CTA take every step together (see coop_lin_kernel)
    for (long b0 = (long)blockIdx.x * wpc; b0 < p.batch; b0 += (long)gridDim.x * wpc) {
        const long b = b0 + team_index<Team>();
        const bool live = b < p.batch;
        if (live) {
            if constexpr (kVaried) varied_row(tt, *v, b, tm);
            for (int i = lane; i < nq; i += TS) {
                const double v = p.q1[b * nq + i];
                w[lay.q1 + i] = v;
                w[lay.q2 + i] = v;
            }
            tm.sync();
            for (int i = lane; i < nd; i += TS) {
                w[lay.p1 + i] = p.p1[b * nd + i];
                if (p.q2g) w[lay.q2 + i] = p.q2g[b * nd + i];
            }
            for (int i = lane; i < nc; i += TS) w[lay.lam + i] = p.lamg ? p.lamg[b * nc + i] : 0.0;
        }
        int total = 0, status = ST_OK;
        double t1 = p.t0;
        for (int s = 0; s < p.nsteps; ++s) {
            TREPB_LOCKSTEP();
            if (!live || status != ST_OK) continue;
            if (s > 0) {
                for (int i = lane; i < nq; i += TS) w[lay.q1 + i] = w[lay.q2 + i];
                for (int i = lane; i < nd; i += TS) w[lay.p1 + i] = w[lay.p2 + i];
            }
            for (int i = lane; i < nu; i += TS) w[lay.u1 + i] = p.u1 ? p.u1[(b * p.nsteps + s) * nu + i] : 0.0;
            tm.sync();
            for (int i = lane; i < nk; i += TS) w[lay.q2 + nd + i] = p.k2[(b * p.nsteps + s) * nk + i];
            tm.sync();
            if (p.times) t1 = p.times[s];
            const double t2 = p.times ? p.times[s + 1] : t1 + p.dt;
            const int it = c.solve(t1, t2, p.tol, p.max_it);
            if (it < 0) { status = it; continue; }
            total += it;
            t1 = t2;
            if (p.sample_every > 0 && (s + 1) % p.sample_every == 0) {
                const long row = b * p.nsamples + (s + 1) / p.sample_every - 1;
                if (p.traj_q) for (int i = lane; i < nq; i += TS) p.traj_q[row * nq + i] = w[lay.q2 + i];
                if (p.traj_p) for (int i = lane; i < nd; i += TS) p.traj_p[row * nd + i] = w[lay.p2 + i];
            }
        }
        tm.sync();
        if (live) {
            for (int i = lane; i < nq; i += TS) p.q2[b * nq + i] = w[lay.q2 + i];
            for (int i = lane; i < nd; i += TS) p.p2[b * nd + i] = w[lay.p2 + i];
            if (p.lam) for (int i = lane; i < nc; i += TS) p.lam[b * nc + i] = w[lay.lam + i];
            if (lane == 0) {
                if (p.iters) p.iters[b] = total;
                p.status[b] = status;
            }
        }
        tm.sync();
    }
}

template <class D, class Team, int TEAMS>
__global__ void __launch_bounds__(TEAMS * Team::kSize, 1)
coop_step_kernel(const CoopSys gs, const int blob_bytes, const CoopLayout lay_, const StepParams p, double* __restrict__ ext) {
    coop_step_body<D, Team, TEAMS, false>(gs, blob_bytes, lay_, p, ext, nullptr);
}
template <class D, class Team, int TEAMS>
__global__ void __launch_bounds__(TEAMS * Team::kSize, 1)
coop_step_varied_kernel(const CoopSys gs, const int blob_bytes, const CoopLayout lay_, const StepParams p, double* __restrict__ ext,
                        const CoopVaried v) {
    coop_step_body<D, Team, TEAMS, true>(gs, blob_bytes, lay_, p, ext, &v);
}

// DSystem.project / armijo_simulate (trep/discopt/dsystem.py:426-457): closed-loop rollouts, one warp per
// candidate, the affine feedback U[k] = bU[k] - K[k](X[k] - bX[k]) evaluated by the lanes (one input
// component each) inside the time loop.
template <class D, class Team, int TEAMS, bool kVaried>
__device__ __forceinline__ void
coop_project_body(const CoopSys& gs, const int blob_bytes, const CoopLayout& lay_, const ProjParams& p, double* __restrict__ ext,
                  const CoopVaried* v) {
    CoopLayout lay = lay_;
    if constexpr (D::kStatic) lay = static_layout<D>(gs, true);
    Stage st = coop_stage<Team>(gs, blob_bytes, lay);
    const Team tm = make_team<Team>();
    TeamTables tt;
    if constexpr (kVaried) varied_init(tt, st, blob_bytes, *v, tm);
    const CoopSys& S = team_sys<kVaried>(st, tt);
    double* w = st.w;
    constexpr int TS = Team::kSize;
    Coop<Team, D> c(S, lay, w, tm, team_slab<D, Team>(ext, lay));
    const int lane = tm.lane(), wpc = blockDim.x / TS;
    const int nd = c.ND(), nk = c.NK(), nq = c.NQ(), nu = c.NU(), nc = c.NC();
    const int nX = 2 * nq, nU = nu + nk, K = p.nsteps;
    for (long b0 = (long)blockIdx.x * wpc; b0 < p.batch; b0 += (long)gridDim.x * wpc) {
        const long b = b0 + team_index<Team>();
        const bool live = b < p.batch;
        const double* bX = p.bX + b * (long)(K + 1) * nX;
        const double* bU = p.bU + b * (long)K * nU;
        const double* Kf = p.K + (p.k_per_instance ? b * (long)K * nU * nX : 0);
        double* Xo = p.X + b * (long)(K + 1) * nX;
        double* Uo = p.U + b * (long)K * nU;
        if (live) {
            if constexpr (kVaried) varied_row(tt, *v, b, tm);
            for (int i = lane; i < nq; i += TS) { const double v = bX[i]; w[lay.q2 + i] = v; Xo[i] = v; }
            for (int i = lane; i < nd; i += TS) { const double v = bX[nq + i]; w[lay.p2 + i] = v; Xo[nq + i] = v; }
            for (int i = lane; i < nk; i += TS) { const double v = bX[nq + nd + i]; w[lay.vk + i] = v; Xo[nq + nd + i] = v; }
            for (int i = lane; i < nc; i += TS) w[lay.lam + i] = 0.0;
        }
        int total = 0, status = ST_OK, fail = K;
        double t1 = p.t0;
        for (int s = 0; s < K; ++s) {
            TREPB_LOCKSTEP();   // the warps of a CTA take every step together (see coop_lin_kernel)
            if (!live || status != ST_OK) continue;
            for (int i = lane; i < nq; i += TS) w[lay.q1 + i] = w[lay.q2 + i];
            for (int i = lane; i < nd; i += TS) w[lay.p1 + i] = w[lay.p2 + i];
            tm.sync();
            const double* bx = bX + (long)s * nX;
            const double* Ks = Kf + (long)s * nU * nX;
            for (int cc = lane; cc < nU; cc += TS) {
                double acc = 0.0;
                for (int x = 0; x < nq; ++x) acc += Ks[cc * nX + x] * (w[lay.q1 + x] - bx[x]);
                for (int x = 0; x < nd; ++x) acc += Ks[cc * nX + nq + x] * (w[lay.p1 + x] - bx[nq + x]);
                for (int x = 0; x < nk; ++x) acc += Ks[cc * nX + nq + nd + x] * (w[lay.vk + x] - bx[nq + nd + x]);
                const double u = bU[(long)s * nU + cc] - acc;
                Uo[(long)s * nU + cc] = u;
                if (cc < nu) w[lay.u1 + cc] = u;
                else w[lay.q2 + nd + cc - nu] = u;
            }
            if (p.use_hint) for (int i = lane; i < nd; i += TS) w[lay.q2 + i] = bX[(long)(s + 1) * nX + i];
            tm.sync();
            if (p.times) t1 = p.times[s];
            const double t2 = p.times ? p.times[s + 1] : t1 + p.dt;
            const int it = c.solve(t1, t2, p.tol, p.max_it);
            if (it < 0) { status = it; fail = s; continue; }
            total += it;
            const double dts = t2 - t1;
            t1 = t2;
            double* xo = Xo + (long)(s + 1) * nX;
            for (int i = lane; i < nq; i += TS) xo[i] = w[lay.q2 + i];
            for (int i = lane; i < nd; i += TS) xo[nq + i] = w[lay.p2 + i];
            for (int i = lane; i < nk; i += TS) {
                const double v = (w[lay.q2 + nd + i] - w[lay.q1 + nd + i]) / dts;
                w[lay.vk + i] = v;
                xo[nq + nd + i] = v;
            }
            tm.sync();
        }
        if (live && lane == 0) {
            if (p.iters) p.iters[b] = total;
            p.status[b] = status;
            if (p.fail_step) p.fail_step[b] = fail;
        }
        tm.sync();
    }
}

template <class D, class Team, int TEAMS>
__global__ void __launch_bounds__(TEAMS * Team::kSize, 1)
coop_project_kernel(const CoopSys gs, const int blob_bytes, const CoopLayout lay_, const ProjParams p, double* __restrict__ ext) {
    coop_project_body<D, Team, TEAMS, false>(gs, blob_bytes, lay_, p, ext, nullptr);
}
template <class D, class Team, int TEAMS>
__global__ void __launch_bounds__(TEAMS * Team::kSize, 1)
coop_project_varied_kernel(const CoopSys gs, const int blob_bytes, const CoopLayout lay_, const ProjParams p,
                           double* __restrict__ ext, const CoopVaried v) {
    coop_project_body<D, Team, TEAMS, true>(gs, blob_bytes, lay_, p, ext, &v);
}

template <class D, class Team, int TEAMS, bool kVaried>
__device__ __forceinline__ void
coop_p2_body(const CoopSys& gs, const int blob_bytes, const CoopLayout& lay_, const P2Params& p, double* __restrict__ ext,
             const CoopVaried* v) {
    CoopLayout lay = lay_;
    if constexpr (D::kStatic) lay = static_layout<D>(gs, true);
    Stage st = coop_stage<Team>(gs, blob_bytes, lay);
    const Team tm = make_team<Team>();
    TeamTables tt;
    if constexpr (kVaried) varied_init(tt, st, blob_bytes, *v, tm);
    const CoopSys& S = team_sys<kVaried>(st, tt);
    double* w = st.w;
    constexpr int TS = Team::kSize;
    Coop<Team, D> c(S, lay, w, tm, team_slab<D, Team>(ext, lay));
    const int lane = tm.lane(), wpc = blockDim.x / TS;
    const int nd = c.ND(), nq = c.NQ(), nu = c.NU(), nc = c.NC();
    for (long b = (long)blockIdx.x * wpc + team_index<Team>(); b < p.batch; b += (long)gridDim.x * wpc) {
        if constexpr (kVaried) varied_row(tt, *v, b, tm);
        for (int i = lane; i < nq; i += TS) {
            w[lay.q1 + i] = p.q0[b * nq + i];
            w[lay.q2 + i] = p.q1[b * nq + i];
        }
        for (int i = lane; i < nu; i += TS) w[lay.u1 + i] = p.u1 ? p.u1[b * nu + i] : 0.0;
        if (p.mode == 1) {
            for (int i = lane; i < nd; i += TS) w[lay.p1 + i] = p.p1[b * nd + i];
            for (int i = lane; i < nc; i += TS) w[lay.lam + i] = p.lam ? p.lam[b * nc + i] : 0.0;
        }
        tm.sync();
        if (p.mode == 0) {
            c.calc_p2(p.dt);
            for (int i = lane; i < nd; i += TS) p.p[b * nd + i] = w[lay.p2 + i];
        } else if (p.mode == 1) {
            c.calc_f(p.dt);
            for (int i = lane; i < nd + nc; i += TS) p.p[b * (nd + nc) + i] = w[lay.fr + i];
        } else {
            c.calc_fm2(p.dt);
            for (int i = lane; i < nd; i += TS) p.p[b * nd + i] = w[lay.fr + i];
        }
        tm.sync();
    }
}

template <class D, class Team, int TEAMS>
__global__ void __launch_bounds__(TEAMS * Team::kSize, 1)
coop_p2_kernel(const CoopSys gs, const int blob_bytes, const CoopLayout lay_, const P2Params p, double* __restrict__ ext) {
    coop_p2_body<D, Team, TEAMS, false>(gs, blob_bytes, lay_, p, ext, nullptr);
}
template <class D, class Team, int TEAMS>
__global__ void __launch_bounds__(TEAMS * Team::kSize, 1)
coop_p2_varied_kernel(const CoopSys gs, const int blob_bytes, const CoopLayout lay_, const P2Params p, double* __restrict__ ext,
                      const CoopVaried v) {
    coop_p2_body<D, Team, TEAMS, true>(gs, blob_bytes, lay_, p, ext, &v);
}

template <class D, class Team, int TEAMS, bool kVaried>
__device__ __forceinline__ void
coop_lin_body(const CoopSys& gs, const int blob_bytes, const CoopLayout& lay_, const LinParams& p, const AuxLayout& al,
              double* __restrict__ ext, const CoopVaried* v) {
    CoopLayout lay = lay_;
    if constexpr (D::kStatic) lay = static_layout<D>(gs, false);
    Stage st = coop_stage<Team>(gs, blob_bytes, lay);
    const Team tm = make_team<Team>();
    TeamTables tt;
    if constexpr (kVaried) varied_init(tt, st, blob_bytes, *v, tm);
    const CoopSys& S = team_sys<kVaried>(st, tt);
    double* w = st.w;
    constexpr int TS = Team::kSize;
    Coop<Team, D> c(S, lay, w, tm, team_slab<D, Team>(ext, lay));
    const int lane = tm.lane(), wpc = blockDim.x / TS;
    const int nd = c.ND(), nk = c.NK(), nq = c.NQ(), nu = c.NU(), nc = c.NC();
    const long nX = 2 * nq, nU = nu + nk, nA = nX * nX, nB = nX * nU;
    const int auxo[7] = {al.o_m2, al.o_m2p, al.o_pj, al.o_pjp, al.o_dh1, al.o_dh2, al.o_t22};
    // The warps of a CTA start every instance together (one __syncthreads per round): the kernel is
    // ~200 KB of SASS, and seven warps drifting through different phases of it miss the instruction
    // cache a third of the time (ncu: "no instruction" stalls 31 % free-running vs 5 % in step); the
    // wait for the slowest Newton iteration count of the round costs less than that.
#pragma unroll 1
    for (long b0 = (long)blockIdx.x * wpc; b0 < p.batch; b0 += (long)gridDim.x * wpc, TREPB_LOCKSTEP()) {
        const long b = b0 + team_index<Team>();
        if (b >= p.batch) continue;
        if constexpr (kVaried) varied_row(tt, *v, p.traj_len > 1 ? b / (p.traj_len - 1) : b, tm);
        const long r = p.traj_len > 1 ? b + b / (p.traj_len - 1) : b;   // state row (trepb_lin_args.traj_len)
        for (int i = lane; i < nq; i += TS) {
            const double v = p.q1[r * nq + i];
            w[lay.q1 + i] = v;
            w[lay.q2 + i] = v;
        }
        tm.sync();
        for (int i = lane; i < nd; i += TS) {
            w[lay.p1 + i] = p.p1[r * nd + i];
            if (p.q2g) w[lay.q2 + i] = p.q2g[r * nd + i];
        }
        for (int i = lane; i < nk; i += TS) w[lay.q2 + nd + i] = p.k2[b * nk + i];
        for (int i = lane; i < nu; i += TS) w[lay.u1 + i] = p.u1[b * nu + i];
        for (int i = lane; i < nc; i += TS) w[lay.lam + i] = p.lamg ? p.lamg[b * nc + i] : 0.0;
        tm.sync();
        const double t1 = p.t1 ? p.t1[b] : p.t1s;
        const double t2 = p.t2 ? p.t2[b] : (t1 + p.dts);
        int it = c.solve(t1, t2, p.tol, p.max_it);
        int status = ST_OK;
        if (it < 0) { status = it; it = 0; }
        tm.sync();
        if (p.q2) for (int i = lane; i < nq; i += TS) p.q2[b * nq + i] = w[lay.q2 + i];
        if (p.p2) for (int i = lane; i < nd; i += TS) p.p2[b * nd + i] = w[lay.p2 + i];
        if (p.lam) for (int i = lane; i < nc; i += TS) p.lam[b * nc + i] = w[lay.lam + i];
        if (status == ST_OK) {
            Deriv1Out o;
#define TREPB_RAW(idx, member, rows, cols) \
            o.member = p.raw[idx] ? p.raw[idx] + b * (long)((rows) * (cols)) : nullptr;
            TREPB_RAW(0, q2_dq1, nq, nd) TREPB_RAW(1, q2_dp1, nd, nd) TREPB_RAW(2, q2_du1, nu, nd) TREPB_RAW(3, q2_dk2, nk, nd)
            TREPB_RAW(4, p2_dq1, nq, nd) TREPB_RAW(5, p2_dp1, nd, nd) TREPB_RAW(6, p2_du1, nu, nd) TREPB_RAW(7, p2_dk2, nk, nd)
            TREPB_RAW(8, l1_dq1, nq, nc) TREPB_RAW(9, l1_dp1, nd, nc) TREPB_RAW(10, l1_du1, nu, nc) TREPB_RAW(11, l1_dk2, nk, nc)
#undef TREPB_RAW
            o.es = 1;
            o.A = p.A ? p.A + b * nA : nullptr;
            o.B = p.B ? p.B + b * nB : nullptr;
            const int r = c.deriv1(t1, t2, o, p.aux ? p.aux + b * (long)p.aux_size : nullptr, auxo);
            if (r < 0) status = r;
        }
        if (lane == 0) {
            if (p.iters) p.iters[b] = it;
            p.status[b] = status;
        }
        tm.sync();
    }
}

template <class D, class Team, int TEAMS>
__global__ void __launch_bounds__(TEAMS * Team::kSize, 1)
coop_lin_kernel(const CoopSys gs, const int blob_bytes, const CoopLayout lay_, const LinParams p, const AuxLayout al,
                double* __restrict__ ext) {
    coop_lin_body<D, Team, TEAMS, false>(gs, blob_bytes, lay_, p, al, ext, nullptr);
}
template <class D, class Team, int TEAMS>
__global__ void __launch_bounds__(TEAMS * Team::kSize, 1)
coop_lin_varied_kernel(const CoopSys gs, const int blob_bytes, const CoopLayout lay_, const LinParams p, const AuxLayout al,
                       double* __restrict__ ext, const CoopVaried v) {
    coop_lin_body<D, Team, TEAMS, true>(gs, blob_bytes, lay_, p, al, ext, &v);
}

template <class K>
cudaError_t prep(K kernel, size_t smem) {
    if (smem > 48 * 1024)
        return cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    return cudaSuccess;
}

// Two instantiations per kernel: the base one (kSolveTeams / kLinTeams teams per CTA, up to 168 / 255 registers
// per thread) and, for shapes whose workspace is small enough that more teams fit in shared memory, a wide one
// (kWideTeamsCt / kWideTeamsRt teams, 128 / 64 registers): these kernels are latency-bound, their throughput grows almost linearly
// with the instances in flight per SM (marionette linearize: 1.41 / 2.73 / 3.82 / 4.92e6 /s at 2 / 4 / 6 / 8).
template <class D>
constexpr bool wide_fits() {
    if constexpr (D::kStatic) return (size_t)D::layout(true).total * 8 * (kSolveTeams + 1) <= 200 * 1024;
    else return true;
}
template <class D, class Team>
struct Launch {
    static constexpr bool kWide = Team::kWarps == 1 && !D::kExt && !D::Solve::kExtS && wide_fits<D>();
    static constexpr int kWideTeams = D::kStatic ? kWideTeamsCt : kWideTeamsRt;
    static constexpr int kLin = D::kExt ? kExtLinTeams : kLinTeams;   // teams per CTA of the base linearize instantiation
    static constexpr int kSolve = D::Solve::kExtS ? kExtSolveTeams : kSolveTeams;   // ... of the step / project / p2 ones
    static cudaError_t step(const CoopLaunch& c, const StepParams& p) {
        if constexpr (kWide) if (c.warps > kSolve) {
            cudaError_t e = prep(coop_step_kernel<typename D::Solve, WarpTeam, kWideTeams>, c.smem);
            if (e != cudaSuccess) return e;
            coop_step_kernel<typename D::Solve, WarpTeam, kWideTeams><<<c.grid, 32 * c.warps, c.smem, c.stream>>>(c.sys, c.blob_bytes, c.lay, p, c.ext);
            return cudaGetLastError();
        }
        cudaError_t e = prep(coop_step_kernel<typename D::Solve, WarpTeam, kSolve>, c.smem);
        if (e != cudaSuccess) return e;
        coop_step_kernel<typename D::Solve, WarpTeam, kSolve><<<c.grid, 32 * c.warps, c.smem, c.stream>>>(c.sys, c.blob_bytes, c.lay, p, c.ext);
        return cudaGetLastError();
    }
    static cudaError_t p2(const CoopLaunch& c, const P2Params& p) {
        if constexpr (kWide) if (c.warps > kSolve) {
            cudaError_t e = prep(coop_p2_kernel<typename D::Solve, WarpTeam, kWideTeams>, c.smem);
            if (e != cudaSuccess) return e;
            coop_p2_kernel<typename D::Solve, WarpTeam, kWideTeams><<<c.grid, 32 * c.warps, c.smem, c.stream>>>(c.sys, c.blob_bytes, c.lay, p, c.ext);
            return cudaGetLastError();
        }
        cudaError_t e = prep(coop_p2_kernel<typename D::Solve, WarpTeam, kSolve>, c.smem);
        if (e != cudaSuccess) return e;
        coop_p2_kernel<typename D::Solve, WarpTeam, kSolve><<<c.grid, 32 * c.warps, c.smem, c.stream>>>(c.sys, c.blob_bytes, c.lay, p, c.ext);
        return cudaGetLastError();
    }
    static cudaError_t lin(const CoopLaunch& c, const LinParams& p, const AuxLayout& al) {
        if constexpr (kWide) if (c.warps > kLin) {
            cudaError_t e = prep(coop_lin_kernel<D, Team, kWideTeams>, c.smem);
            if (e != cudaSuccess) return e;
            coop_lin_kernel<D, Team, kWideTeams><<<c.grid, Team::kSize * c.warps, c.smem, c.stream>>>(c.sys, c.blob_bytes, c.lay, p, al, c.ext);
            return cudaGetLastError();
        }
        cudaError_t e = prep(coop_lin_kernel<D, Team, kLin>, c.smem);
        if (e != cudaSuccess) return e;
        coop_lin_kernel<D, Team, kLin><<<c.grid, Team::kSize * c.warps, c.smem, c.stream>>>(c.sys, c.blob_bytes, c.lay, p, al, c.ext);
        return cudaGetLastError();
    }
    static cudaError_t proj(const CoopLaunch& c, const ProjParams& p) {
        if constexpr (kWide) if (c.warps > kSolve) {
            cudaError_t e = prep(coop_project_kernel<typename D::Solve, WarpTeam, kWideTeams>, c.smem);
            if (e != cudaSuccess) return e;
            coop_project_kernel<typename D::Solve, WarpTeam, kWideTeams><<<c.grid, 32 * c.warps, c.smem, c.stream>>>(c.sys, c.blob_bytes, c.lay, p, c.ext);
            return cudaGetLastError();
        }
        cudaError_t e = prep(coop_project_kernel<typename D::Solve, WarpTeam, kSolve>, c.smem);
        if (e != cudaSuccess) return e;
        coop_project_kernel<typename D::Solve, WarpTeam, kSolve><<<c.grid, 32 * c.warps, c.smem, c.stream>>>(c.sys, c.blob_bytes, c.lay, p, c.ext);
        return cudaGetLastError();
    }
    template <class K, class... A>
    static cudaError_t go(K kernel, const CoopLaunch& c, int threads, const A&... args) {
        cudaError_t e = prep(kernel, c.smem);
        if (e != cudaSuccess) return e;
        kernel<<<c.grid, threads, c.smem, c.stream>>>(args...);
        return cudaGetLastError();
    }
    // per-instance parameters: the varied instantiations, selected as above
    static cudaError_t step_v(const CoopLaunch& c, const StepParams& p, const CoopVaried& v) {
        if constexpr (kWide) if (c.warps > kSolve)
            return go(coop_step_varied_kernel<typename D::Solve, WarpTeam, kWideTeams>, c, 32 * c.warps, c.sys, c.blob_bytes, c.lay, p, c.ext, v);
        return go(coop_step_varied_kernel<typename D::Solve, WarpTeam, kSolve>, c, 32 * c.warps, c.sys, c.blob_bytes, c.lay, p, c.ext, v);
    }
    static cudaError_t p2_v(const CoopLaunch& c, const P2Params& p, const CoopVaried& v) {
        if constexpr (kWide) if (c.warps > kSolve)
            return go(coop_p2_varied_kernel<typename D::Solve, WarpTeam, kWideTeams>, c, 32 * c.warps, c.sys, c.blob_bytes, c.lay, p, c.ext, v);
        return go(coop_p2_varied_kernel<typename D::Solve, WarpTeam, kSolve>, c, 32 * c.warps, c.sys, c.blob_bytes, c.lay, p, c.ext, v);
    }
    static cudaError_t lin_v(const CoopLaunch& c, const LinParams& p, const AuxLayout& al, const CoopVaried& v) {
        if constexpr (kWide) if (c.warps > kLin)
            return go(coop_lin_varied_kernel<D, Team, kWideTeams>, c, Team::kSize * c.warps, c.sys, c.blob_bytes, c.lay, p, al, c.ext, v);
        return go(coop_lin_varied_kernel<D, Team, kLin>, c, Team::kSize * c.warps, c.sys, c.blob_bytes, c.lay, p, al, c.ext, v);
    }
    static cudaError_t proj_v(const CoopLaunch& c, const ProjParams& p, const CoopVaried& v) {
        if constexpr (kWide) if (c.warps > kSolve)
            return go(coop_project_varied_kernel<typename D::Solve, WarpTeam, kWideTeams>, c, 32 * c.warps, c.sys, c.blob_bytes, c.lay, p, c.ext, v);
        return go(coop_project_varied_kernel<typename D::Solve, WarpTeam, kSolve>, c, 32 * c.warps, c.sys, c.blob_bytes, c.lay, p, c.ext, v);
    }
    // which: 0 step, 1 p2, 2 lin, 3 project; + 4 for the wide instantiation
    static cudaError_t info(int which, KernelInfo* ki) {
        const void* fn = nullptr;
        if (which >= 4) {
            if constexpr (kWide) {
                fn = which == 4 ? (const void*)coop_step_kernel<typename D::Solve, WarpTeam, kWideTeams>
                   : which == 5 ? (const void*)coop_p2_kernel<typename D::Solve, WarpTeam, kWideTeams>
                   : which == 6 ? (const void*)coop_lin_kernel<D, Team, kWideTeams> : (const void*)coop_project_kernel<typename D::Solve, WarpTeam, kWideTeams>;
            } else {
                return cudaErrorInvalidValue;
            }
        } else {
            fn = which == 0 ? (const void*)coop_step_kernel<typename D::Solve, WarpTeam, kSolve>
               : which == 1 ? (const void*)coop_p2_kernel<typename D::Solve, WarpTeam, kSolve>
               : which == 2 ? (const void*)coop_lin_kernel<D, Team, kLin> : (const void*)coop_project_kernel<typename D::Solve, WarpTeam, kSolve>;
        }
        cudaFuncAttributes a;
        cudaError_t e = cudaFuncGetAttributes(&a, fn);
        if (e != cudaSuccess) return e;
        ki->regs = a.numRegs;
        ki->max_threads = a.maxThreadsPerBlock;
        ki->static_smem = a.sharedSizeBytes;
        ki->local_bytes = a.localSizeBytes;
        return cudaSuccess;
    }
    static bool matches(const CoopSys& s) {
        if constexpr (D::kStatic) return D::matches(s);
        else return true;
    }
};

}  // namespace coopk

template <class D, class Team = WarpTeam>
CoopKernelSet make_coop_kernelset(const char* name) {
    CoopKernelSet k;
    k.name = name;
    k.specialized = D::kStatic ? 1 : 0;
    k.team_warps = Team::kWarps;
    k.max_teams = coopk::Launch<D, Team>::kWide ? coopk::Launch<D, Team>::kWideTeams : 0;
    k.lin_teams = coopk::Launch<D, Team>::kLin;
    k.solve_teams = coopk::Launch<D, Team>::kSolve;
    k.ext = D::kExt ? 1 : 0;
    k.matches = &coopk::Launch<D, Team>::matches;
    k.step = &coopk::Launch<D, Team>::step;
    k.p2 = &coopk::Launch<D, Team>::p2;
    k.lin = &coopk::Launch<D, Team>::lin;
    k.proj = &coopk::Launch<D, Team>::proj;
    k.info = &coopk::Launch<D, Team>::info;
    k.step_v = &coopk::Launch<D, Team>::step_v;
    k.p2_v = &coopk::Launch<D, Team>::p2_v;
    k.lin_v = &coopk::Launch<D, Team>::lin_v;
    k.proj_v = &coopk::Launch<D, Team>::proj_v;
    return k;
}

}  // namespace trepb
