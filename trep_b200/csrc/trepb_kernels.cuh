// CUDA kernels of the batched MidpointVI path (sm_100a, fp64): one thread per instance.
//
//   step_kernel       trepb_step_batch*      == MidpointVI.step looped in-kernel
//                                               (trep/midpointvi.py:174-201 -> midpointvi.c:691-747)
//   p2_kernel         trepb_calc_p2_batch*   == MidpointVI.calc_p2 (midpointvi.c:491-504)
//   linearize_kernel  trepb_linearize_batch* == solve_DEL + calc_deriv1 + DSystem.fdx/fdu
//                                               (midpointvi.c:1100-1120, dsystem.py:284-317)
//
// The same kernel templates are instantiated
//   * on RtSys + WsStrided  - the table-driven general path: the packed system description is
//     staged into shared memory once per CTA, the per-instance workspace lives in a global slab
//     laid out [element][thread] so every workspace access of a warp is one coalesced line;
//   * on a generated constexpr system + WsStatic - the specialised path for small systems: all
//     loops unrolled, workspace in registers, no table reads at all.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "trepb_hd.h"
#include "trepb_math.cuh"
#include "trepb_varied.h"

namespace trepb {

struct StepParams {
    long long batch;
    int nsteps, max_it;
    double t0, dt, tol;
    double tolT;      // sqrt_threshold(tol), computed on the host
    const double *q1, *p1, *u1, *k2, *q2g, *lamg;
    double *q2, *p2, *lam;
    int *iters, *status;
    int sample_every, nsamples;
    double *traj_q, *traj_p;
    const double* times;   // [nsteps+1] or null
};

// closed-loop rollouts (trepb_project_batch*)
struct ProjParams {
    long long batch;
    int nsteps, max_it;
    double t0, dt, tol;
    double tolT;      // sqrt_threshold(tol), computed on the host
    const double *bX, *bU, *K;
    int k_per_instance, use_hint;
    double *X, *U;
    int *iters, *status, *fail_step;
    const double* times;   // [nsteps+1] or null
};

struct P2Params {
    long long batch;
    double dt;
    const double *q0, *q1;
    double* p;
    // mode 0: p2 (calc_p2); 1: residual f [nd+nc] (MidpointVI_calc_f); 2: fm2 [nd] (discrete_fm2)
    int mode;
    const double *p1, *u1, *lam;
};

struct LinParams {
    long long batch;
    int max_it;
    double tol, t1s, dts;
    double tolT;      // sqrt_threshold(tol), computed on the host
    const double *t1, *t2;
    const double *q1, *p1, *u1, *k2, *q2g, *lamg;
    double *q2, *p2, *lam;
    int *iters, *status;
    double *A, *B;
    double* raw[12];  // q2_dq1 q2_dp1 q2_du1 q2_dk2 p2_d* l1_d*
    int stage;        // 1: stage A/B through shared memory for coalesced stores
    int traj_len;     // 0, or rows per state trajectory (instance b reads state row b + b / (traj_len - 1))
    double* aux;      // [B][AuxLayout::size] factorizations for the second-derivative kernel, or null
    int aux_size;
};

// per-instance data exported by the linearize kernel for this kernel
struct AuxLayout {
    int o_m2, o_m2p, o_pj, o_pjp, o_dh1, o_dh2, o_t22, size;
    TREPB_HD void set(int nd, int nc) {
        int o = 0;
        o_m2 = o; o += nd * nd;
        o_m2p = o; o += nd;
        o_pj = o; o += nc * nc;
        o_pjp = o; o += nc;
        o_dh1 = o; o += nc * nd;
        o_dh2 = o; o += nc * nd;
        o_t22 = o; o += nd * nd;
        size = o;
    }
};

struct D2Params {
    long long batch;
    int nx, npairs;
    double t1s, dts;
    const double *t1, *t2;
    const double *q1, *u1;          // inputs of the step            [B][nq], [B][nu]
    const double *q2, *lam;         // converged step                [B][nq], [B][nc]
    const double* q2_d[4];          // deriv1, [B][wrt][nd]   (dq1, dp1, du1, dk2)
    const double* l1_d[4];          // deriv1, [B][wrt][nc]
    const double* aux;              // [B][aux.size]
    AuxLayout auxl;
    const int* status;              // instances whose step/deriv1 failed are skipped
    double* out[3][10];             // q2 / p2 / l1  x  pair kind ; any may be null
    const double* z;                // [B][nX] or null: z-contracted outputs (DSystem.fdxdx(z) ...)
    double *zxx, *zxu, *zuu;        // [B][nX][nX], [B][nX][nU], [B][nU][nU] (pre-zeroed)
};


// What a kernel launch needs besides its parameters.
struct LaunchCfg {
    int grid, block;
    size_t smem;
    cudaStream_t stream;
    const RtSys* sys;       // host copy of the device view (general path); ignored when specialised
    const char* dblob;      // device address of the packed blob
    int blob_bytes;
    WsStrided ws;           // workspace slab view (general path)
    const double* spec_params;   // host: run-time parameters of a specialised system (trepb::param_map order)
};

struct KernelInfo {
    int regs, max_threads;
    size_t static_smem, local_bytes;
};

struct KernelSet {
    const char* name;
    unsigned long long hash;  // 0: general
    int specialized;
    int nX, nU;
    int n_params;            // specialised: number of run-time parameters the kernels take (param_map order)
    // per-instance parameters (trepb_*_varied_batch*): a non-null VariedArgs launches the same kernel body
    // instantiated with kVaried (*_varied_kernel)
    cudaError_t (*step)(const LaunchCfg&, const StepParams&, const VariedArgs*);
    cudaError_t (*p2)(const LaunchCfg&, const P2Params&, const VariedArgs*);
    cudaError_t (*lin)(const LaunchCfg&, const LinParams&, const VariedArgs*);
    cudaError_t (*proj)(const LaunchCfg&, const ProjParams&, const VariedArgs*);
    // which: 0 step, 1 p2, 2 lin, 3 project, of the *_varied_kernel set when `varied`.  blocks_per_sm at (block, smem).
    cudaError_t (*occupancy)(int which, bool varied, int block, size_t smem, int* blocks_per_sm, KernelInfo* info);
    // second derivatives, per-pair scheme: d2_kernel, or d2_varied_kernel for a non-null VariedArgs / `varied`
    cudaError_t (*d2)(const LaunchCfg&, const WsStridedT<HDG>&, const D2Params&, const VariedArgs*);
    cudaError_t (*d2_occupancy)(bool varied, int block, size_t smem, int* blocks_per_sm, KernelInfo* info);
};

// factorizations and tables of deriv1 that the second-derivative kernel reuses (AuxLayout)
template <class Sys, class Ws>
TREPB_HD void export_aux(const Sys& sys, Ws& ws, double* ax) {
    const int nd = sys.ND(), nc = sys.NC();
    AuxLayout al;
    al.set(nd, nc);
    TREPB_UNROLL_SYS
    for (int i = 0; i < nd; ++i) {
        ax[al.o_m2p + i] = ws.M2p(i);
        TREPB_UNROLL_SYS
        for (int j = 0; j < nd; ++j) {
            ax[al.o_m2 + i * nd + j] = ws.M2(i, j);
            ax[al.o_t22 + i * nd + j] = ws.T22(i, j);
        }
    }
    TREPB_UNROLL_SYS
    for (int cc = 0; cc < nc; ++cc) {
        ax[al.o_pjp + cc] = ws.PJp(cc);
        TREPB_UNROLL_SYS
        for (int c2 = 0; c2 < nc; ++c2) ax[al.o_pj + cc * nc + c2] = ws.PJ(cc, c2);
        TREPB_UNROLL_SYS
        for (int j = 0; j < nd; ++j) {
            ax[al.o_dh1 + cc * nd + j] = ws.Dh1(cc, j);
            ax[al.o_dh2 + cc * nd + j] = ws.Dh2(cc, j);
        }
    }
}

// registry of ahead-of-time specialised systems (filled by static initialisers of gen/*.cu)
struct SpecRegistry {
    static constexpr int kMax = 64;
    const KernelSet* sets[kMax];
    int n;
};
SpecRegistry& spec_registry();
// Layout fingerprint of everything a specialisation unit shares with the library (kernel parameter structs,
// the kernel-set table).  A plug-in compiled against other headers registers with another fingerprint and is
// refused by spec_register (which lives in the library), instead of being called with mismatched structs.  The base
// constant changes whenever a member of KernelSet changes meaning without changing size (0x30000: d2 / d2_occupancy
// gained their per-instance-parameter argument).
constexpr unsigned kSpecAbi = 0x30000u + (unsigned)(sizeof(RtSys) * 131 + sizeof(StepParams) * 31 + sizeof(LinParams) * 17 +
                                                    sizeof(ProjParams) * 13 + sizeof(P2Params) * 7 + sizeof(D2Params) * 5 +
                                                    sizeof(LaunchCfg) * 3 + sizeof(KernelSet));
bool spec_register(const KernelSet* ks, unsigned abi);
struct SpecRegistrar {
    explicit SpecRegistrar(const KernelSet* ks) { spec_register(ks, kSpecAbi); }
};
const KernelSet* general_kernels();

#if defined(__CUDACC__)
// minimum resident CTAs per SM requested from the compiler (register cap = 65536 / (128 * N));
// experiments: -DTREPB_LB_MIN=6 ...
#ifndef TREPB_LB_MIN
#define TREPB_LB_MIN 0
#endif
// Small specialised systems (<= 2 configs) are asked for 4 resident CTAs per SM (<= 128 registers): measured on
// pend-on-cart's linearize kernel 0.410 -> 0.359 ms per 2^22 instances (130 -> 120 registers, no spills; 5 CTAs
// at 96 registers: 0.369), damped pendulum step 0.746 -> 0.734 ms.  Larger specialised systems keep the whole
// register file per thread (their workspace lives in registers), the table-driven kernels are unconstrained.
// The linearize kernel of those systems streams 224+ bytes per instance and gains from one more CTA: along
// trajectories with exact hints (W3) 1.85e10 linearizations/s at 4 CTAs, 2.04e10 at 5 (96 registers, 44 bytes
// of spills), 1.96e10 at 6; on random states (2.2 Newton iterations) 1.18e10 / 1.14e10 / 1.12e10.
template <class Sys, bool kLin = false>
constexpr int lb_min() {
    if (TREPB_LB_MIN > 0) return TREPB_LB_MIN;
    if constexpr (Sys::kStatic) return Sys::kNQ <= 2 ? (kLin ? 5 : 4) : 1;
    else return 1;
}
// ---------------------------------------------------------------------------------------------
template <class Sys, bool S = Sys::kStatic>
struct Ctx;

// specialised: system is a type, workspace is a local object
template <class Sys>
struct Ctx<Sys, true> {
    using WsT = WsStatic<Sys>;
    Sys sys;
    WsT ws;
    __device__ __forceinline__ Ctx(const RtSys&, const char*, int, const WsStrided&, long, long,
                                   const typename Sys::Params& par) { sys.par = par; }
};

// general: tables staged in shared memory, strided workspace
template <class Sys>
struct Ctx<Sys, false> {
    using WsT = WsStrided;
    RtSys sys;
    WsT ws;
    __device__ __forceinline__ Ctx(const RtSys& s, const char* dblob, int blob_bytes, const WsStrided& w,
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

// kVaried: instance b runs on row `row` of the per-instance parameters (trepb_varied.h).  Specialised: every slot of
// sys.par with a compile-time index, so that the parameters stay in registers; table-driven: the numeric tables
// re-pointed at this thread's expanded slot.
template <class Sys, bool kVaried, class C>
__device__ __forceinline__ void load_params(C& c, const VariedArgs& va, long row, long tid) {
    if constexpr (kVaried) {
        const double* r = va.values + row * va.map.n;
        if constexpr (Sys::kStatic) {
#pragma unroll
            for (int i = 0; i < Sys::kNPAR; ++i) c.sys.par.v[i] = varied_value(va.map, r, i);
        } else {
            varied_point(c.sys, va.map, r, va.slots + tid * (long)va.map.n_out);
        }
    }
}

template <class Sys, bool kVaried>
__device__ __forceinline__ void
step_body(const RtSys& rsys, const char* dblob, int blob_bytes, const WsStrided& wsp, const StepParams& p,
          const typename Sys::Params& par, const VariedArgs& va) {
    const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long nth = (long)gridDim.x * blockDim.x;
    Ctx<Sys> c(rsys, dblob, blob_bytes, wsp, tid, nth, par);
    auto& sys = c.sys;
    auto& ws = c.ws;
    const int nd = sys.ND(), nk = sys.NK(), nq = nd + nk, nu = sys.NU(), nc = sys.NC();
    const double tolT = p.tolT;   // the Newton convergence test needs no square root (sqrt_threshold)
    for (long b = tid; b < p.batch; b += nth) {
        load_params<Sys, kVaried>(c, va, b, tid);
        TREPB_UNROLL_SYS
        for (int i = 0; i < nq; ++i) {
            const double v = p.q1[b * nq + i];
            ws.q1(i) = v;
            ws.q2(i) = v;
        }
        TREPB_UNROLL_SYS
        for (int i = 0; i < nd; ++i) {
            ws.p1(i) = p.p1[b * nd + i];
            if (p.q2g) ws.q2(i) = p.q2g[b * nd + i];
        }
        TREPB_UNROLL_SYS
        for (int i = 0; i < nc; ++i) ws.lam(i) = p.lamg ? p.lamg[b * nc + i] : 0.0;
        int total = 0, status = ST_OK;
        double t1 = p.t0;
        for (int st = 0; st < p.nsteps; ++st) {
            if (st > 0) {
                TREPB_UNROLL_SYS
                for (int i = 0; i < nq; ++i) ws.q1(i) = ws.q2(i);
                TREPB_UNROLL_SYS
                for (int i = 0; i < nd; ++i) ws.p1(i) = ws.p2(i);
            }
            TREPB_UNROLL_SYS
            for (int i = 0; i < nu; ++i) ws.u1(i) = p.u1 ? p.u1[(b * p.nsteps + st) * nu + i] : 0.0;
            TREPB_UNROLL_SYS
            for (int i = 0; i < nk; ++i) ws.q2(nd + i) = p.k2[(b * p.nsteps + st) * nk + i];
            if (p.times) t1 = p.times[st];
            const double t2 = p.times ? p.times[st + 1] : t1 + p.dt;
            const int it = solve_del(sys, ws, t1, t2, p.tol, p.max_it, tolT);
            if (it < 0) { status = it; break; }
            total += it;
            t1 = t2;
            if (p.sample_every > 0 && (st + 1) % p.sample_every == 0) {
                const long row = b * p.nsamples + (st + 1) / p.sample_every - 1;
                if (p.traj_q) {
                    TREPB_UNROLL_SYS
                    for (int i = 0; i < nq; ++i) p.traj_q[row * nq + i] = ws.q2(i);
                }
                if (p.traj_p) {
                    TREPB_UNROLL_SYS
                    for (int i = 0; i < nd; ++i) p.traj_p[row * nd + i] = ws.p2(i);
                }
            }
        }
        TREPB_UNROLL_SYS
        for (int i = 0; i < nq; ++i) p.q2[b * nq + i] = ws.q2(i);
        TREPB_UNROLL_SYS
        for (int i = 0; i < nd; ++i) p.p2[b * nd + i] = ws.p2(i);
        if (p.lam) {
            TREPB_UNROLL_SYS
            for (int i = 0; i < nc; ++i) p.lam[b * nc + i] = ws.lam(i);
        }
        if (p.iters) p.iters[b] = total;
        p.status[b] = status;
    }
}

template <class Sys>
__global__ void __launch_bounds__(128, lb_min<Sys>())
step_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStrided wsp, const StepParams p,
            const typename Sys::Params par) {
    step_body<Sys, false>(rsys, dblob, blob_bytes, wsp, p, par, VariedArgs{});
}
template <class Sys>
__global__ void __launch_bounds__(128, lb_min<Sys>())
step_varied_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStrided wsp, const StepParams p,
                   const VariedArgs va) {
    step_body<Sys, true>(rsys, dblob, blob_bytes, wsp, p, typename Sys::Params{}, va);
}

// DSystem.project / armijo_simulate: X[0] = bX[0]; U[k] = bU[k] - K[k](X[k] - bX[k]); X[k+1] = f(X[k],U[k])
// (trep/discopt/dsystem.py:426-457), one thread per candidate, the feedback inside the time loop.
template <class Sys, bool kVaried>
__device__ __forceinline__ void
project_body(const RtSys& rsys, const char* dblob, int blob_bytes, const WsStrided& wsp, const ProjParams& p,
             const typename Sys::Params& par, const VariedArgs& va) {
    const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long nth = (long)gridDim.x * blockDim.x;
    Ctx<Sys> c(rsys, dblob, blob_bytes, wsp, tid, nth, par);
    auto& sys = c.sys;
    auto& ws = c.ws;
    const int nd = sys.ND(), nk = sys.NK(), nq = nd + nk, nu = sys.NU(), nc = sys.NC();
    const double tolT = p.tolT;   // the Newton convergence test needs no square root (sqrt_threshold)
    const int nX = 2 * nq, nU = nu + nk, K = p.nsteps;
    for (long b = tid; b < p.batch; b += nth) {
        load_params<Sys, kVaried>(c, va, b, tid);
        const double* bX = p.bX + b * (long)(K + 1) * nX;
        const double* bU = p.bU + b * (long)K * nU;
        const double* Kf = p.K + (p.k_per_instance ? b * (long)K * nU * nX : 0);
        double* Xo = p.X + b * (long)(K + 1) * nX;
        double* Uo = p.U + b * (long)K * nU;
        TREPB_UNROLL_SYS for (int i = 0; i < nq; ++i) { const double v = bX[i]; ws.q2(i) = v; Xo[i] = v; }
        TREPB_UNROLL_SYS for (int i = 0; i < nd; ++i) { const double v = bX[nq + i]; ws.p2(i) = v; Xo[nq + i] = v; }
        TREPB_UNROLL_SYS for (int i = 0; i < nk; ++i) { const double v = bX[nq + nd + i]; ws.vk(i) = v; Xo[nq + nd + i] = v; }
        TREPB_UNROLL_SYS for (int i = 0; i < nc; ++i) ws.lam(i) = 0.0;   // set(): initialize_from_state zeroes lambda
        int total = 0, status = ST_OK, fail = K;
        double t1 = p.t0;
        for (int s = 0; s < K; ++s) {
            TREPB_UNROLL_SYS for (int i = 0; i < nq; ++i) ws.q1(i) = ws.q2(i);
            TREPB_UNROLL_SYS for (int i = 0; i < nd; ++i) ws.p1(i) = ws.p2(i);
            const double* bx = bX + (long)s * nX;
            const double* Ks = Kf + (long)s * nU * nX;
            TREPB_UNROLL_SYS
            for (int cc = 0; cc < nU; ++cc) {
                double acc = 0.0;
                TREPB_UNROLL_SYS for (int x = 0; x < nq; ++x) acc += Ks[cc * nX + x] * (ws.q1(x) - bx[x]);
                TREPB_UNROLL_SYS for (int x = 0; x < nd; ++x) acc += Ks[cc * nX + nq + x] * (ws.p1(x) - bx[nq + x]);
                TREPB_UNROLL_SYS for (int x = 0; x < nk; ++x) acc += Ks[cc * nX + nq + nd + x] * (ws.vk(x) - bx[nq + nd + x]);
                const double u = bU[(long)s * nU + cc] - acc;
                Uo[(long)s * nU + cc] = u;
                if (cc < nu) ws.u1(cc) = u;
                else ws.q2(nd + cc - nu) = u;
            }
            if (p.use_hint) { TREPB_UNROLL_SYS for (int i = 0; i < nd; ++i) ws.q2(i) = bX[(long)(s + 1) * nX + i]; }
            if (p.times) t1 = p.times[s];
            const double t2 = p.times ? p.times[s + 1] : t1 + p.dt;
            const int it = solve_del(sys, ws, t1, t2, p.tol, p.max_it, tolT);
            if (it < 0) { status = it; fail = s; break; }
            total += it;
            const double dts = t2 - t1;
            t1 = t2;
            double* xo = Xo + (long)(s + 1) * nX;
            TREPB_UNROLL_SYS for (int i = 0; i < nq; ++i) xo[i] = ws.q2(i);
            TREPB_UNROLL_SYS for (int i = 0; i < nd; ++i) xo[nq + i] = ws.p2(i);
            TREPB_UNROLL_SYS
            for (int i = 0; i < nk; ++i) {
                const double v = (ws.q2(nd + i) - ws.q1(nd + i)) / dts;
                ws.vk(i) = v;
                xo[nq + nd + i] = v;
            }
        }
        if (p.iters) p.iters[b] = total;
        p.status[b] = status;
        if (p.fail_step) p.fail_step[b] = fail;
    }
}

template <class Sys>
__global__ void __launch_bounds__(128, lb_min<Sys>())
project_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStrided wsp, const ProjParams p,
            const typename Sys::Params par) {
    project_body<Sys, false>(rsys, dblob, blob_bytes, wsp, p, par, VariedArgs{});
}
template <class Sys>
__global__ void __launch_bounds__(128, lb_min<Sys>())
project_varied_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStrided wsp, const ProjParams p,
                      const VariedArgs va) {
    project_body<Sys, true>(rsys, dblob, blob_bytes, wsp, p, typename Sys::Params{}, va);
}

template <class Sys, bool kVaried>
__device__ __forceinline__ void
p2_body(const RtSys& rsys, const char* dblob, int blob_bytes, const WsStrided& wsp, const P2Params& p,
        const typename Sys::Params& par, const VariedArgs& va) {
    const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long nth = (long)gridDim.x * blockDim.x;
    Ctx<Sys> c(rsys, dblob, blob_bytes, wsp, tid, nth, par);
    auto& sys = c.sys;
    auto& ws = c.ws;
    const int nd = sys.ND(), nq = sys.NQ(), nu = sys.NU(), nc = sys.NC();
    for (long b = tid; b < p.batch; b += nth) {
        load_params<Sys, kVaried>(c, va, b, tid);
        TREPB_UNROLL_SYS
        for (int i = 0; i < nq; ++i) {
            ws.q1(i) = p.q0[b * nq + i];
            ws.q2(i) = p.q1[b * nq + i];
        }
        TREPB_UNROLL_SYS
        for (int i = 0; i < nu; ++i) ws.u1(i) = p.u1 ? p.u1[b * nu + i] : 0.0;
        if (p.mode == 0) {
            calc_p2(sys, ws, 0.0, p.dt);
            TREPB_UNROLL_SYS
            for (int i = 0; i < nd; ++i) p.p[b * nd + i] = ws.p2(i);
        } else if (p.mode == 1) {
            TREPB_UNROLL_SYS for (int i = 0; i < nd; ++i) ws.p1(i) = p.p1[b * nd + i];
            TREPB_UNROLL_SYS for (int i = 0; i < nc; ++i) ws.lam(i) = p.lam ? p.lam[b * nc + i] : 0.0;
            calc_f(sys, ws, 0.0, p.dt);
            TREPB_UNROLL_SYS
            for (int i = 0; i < nd + nc; ++i) p.p[b * (nd + nc) + i] = ws.fr(i);
        } else {
            eval_mid(sys, ws, Dt(p.dt), 1);
            TREPB_UNROLL_SYS
            for (int i = 0; i < nd; ++i) p.p[b * nd + i] = p.dt * ws.Fo(i);
        }
    }
}

template <class Sys>
__global__ void __launch_bounds__(128)
p2_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStrided wsp, const P2Params p,
            const typename Sys::Params par) {
    p2_body<Sys, false>(rsys, dblob, blob_bytes, wsp, p, par, VariedArgs{});
}
template <class Sys>
__global__ void __launch_bounds__(128)
p2_varied_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStrided wsp, const P2Params p,
                 const VariedArgs va) {
    p2_body<Sys, true>(rsys, dblob, blob_bytes, wsp, p, typename Sys::Params{}, va);
}

template <class Sys, bool kVaried>
__device__ __forceinline__ void
lin_body(const RtSys& rsys, const char* dblob, int blob_bytes, const WsStrided& wsp, const LinParams& p,
         const typename Sys::Params& par, const VariedArgs& va) {
    const long tid = (long)blockIdx.x * blockDim.x + threadIdx.x;
    const long nth = (long)gridDim.x * blockDim.x;
    Ctx<Sys> c(rsys, dblob, blob_bytes, wsp, tid, nth, par);
    auto& sys = c.sys;
    auto& ws = c.ws;
    const int nd = sys.ND(), nk = sys.NK(), nq = nd + nk, nu = sys.NU(), nc = sys.NC();
    const double tolT = p.tolT;   // the Newton convergence test needs no square root (sqrt_threshold)
    const int nX = 2 * nq, nU = nu + nk, nA = nX * nX, nB = nX * nU;
    extern __shared__ double smem_[];
    // loop bound is uniform per warp so that the staged stores can be warp-cooperative
    const long bend = ((p.batch + 31) / 32) * 32;
    for (long b = tid; b < bend; b += nth) {
        const bool live = b < p.batch;
        int it = 0, status = ST_OK;
        Deriv1Out o;
        double t1 = 0.0, t2 = 0.0;
        if (live) {
            const long r = p.traj_len > 1 ? b + b / (p.traj_len - 1) : b;   // input row (see trepb_lin_args.traj_len)
            load_params<Sys, kVaried>(c, va, p.traj_len > 1 ? b / (p.traj_len - 1) : b, tid);   // one row per trajectory
            TREPB_UNROLL_SYS
            for (int i = 0; i < nq; ++i) {
                const double v = p.q1[r * nq + i];
                ws.q1(i) = v;
                ws.q2(i) = v;
            }
            TREPB_UNROLL_SYS
            for (int i = 0; i < nd; ++i) {
                ws.p1(i) = p.p1[r * nd + i];
                if (p.q2g) ws.q2(i) = p.q2g[r * nd + i];
            }
            TREPB_UNROLL_SYS
            for (int i = 0; i < nk; ++i) ws.q2(nd + i) = p.k2[b * nk + i];
            TREPB_UNROLL_SYS
            for (int i = 0; i < nu; ++i) ws.u1(i) = p.u1[b * nu + i];
            TREPB_UNROLL_SYS
            for (int i = 0; i < nc; ++i) ws.lam(i) = p.lamg ? p.lamg[b * nc + i] : 0.0;
            t1 = p.t1 ? p.t1[b] : p.t1s;
            t2 = p.t2 ? p.t2[b] : (t1 + p.dts);
            it = solve_del(sys, ws, t1, t2, p.tol, p.max_it, tolT);
            if (it < 0) { status = it; it = 0; }
            if (p.q2) {
                TREPB_UNROLL_SYS
                for (int i = 0; i < nq; ++i) p.q2[b * nq + i] = ws.q2(i);
            }
            if (p.p2) {
                TREPB_UNROLL_SYS
                for (int i = 0; i < nd; ++i) p.p2[b * nd + i] = ws.p2(i);
            }
            if (p.lam) {
                TREPB_UNROLL_SYS
                for (int i = 0; i < nc; ++i) p.lam[b * nc + i] = ws.lam(i);
            }
        }
#define TREPB_RAW(idx, member, rows, cols) \
        o.member = p.raw[idx] ? p.raw[idx] + b * (long)((rows) * (cols)) : nullptr;
        TREPB_RAW(0, q2_dq1, nq, nd) TREPB_RAW(1, q2_dp1, nd, nd) TREPB_RAW(2, q2_du1, nu, nd) TREPB_RAW(3, q2_dk2, nk, nd)
        TREPB_RAW(4, p2_dq1, nq, nd) TREPB_RAW(5, p2_dp1, nd, nd) TREPB_RAW(6, p2_du1, nu, nd) TREPB_RAW(7, p2_dk2, nk, nd)
        TREPB_RAW(8, l1_dq1, nq, nc) TREPB_RAW(9, l1_dp1, nd, nc) TREPB_RAW(10, l1_du1, nu, nc) TREPB_RAW(11, l1_dk2, nk, nc)
#undef TREPB_RAW
        o.es = 1;
        if (p.stage) {
            // thread-private slot of the CTA tile; stride nA+nB keeps the A and B rows of one
            // instance together
            double* slot = smem_ + (long)threadIdx.x * (nA + nB);
            o.A = p.A ? slot : nullptr;
            o.B = p.B ? slot + nA : nullptr;
        } else {
            o.A = p.A ? p.A + b * nA : nullptr;
            o.B = p.B ? p.B + b * nB : nullptr;
        }
        if (live && status == ST_OK) {
            const int r = deriv1(sys, ws, t1, t2, o, true);
            if (r < 0) status = r;
        }
        if (live && status == ST_OK && p.aux) export_aux(sys, ws, p.aux + b * (long)p.aux_size);
        if (live) {
            if (p.iters) p.iters[b] = it;
            p.status[b] = status;
        }
        if (p.stage) {
            // warp-cooperative coalesced copy: the 32 instances of a warp are contiguous in A and B
            __syncwarp();
            const int lane = threadIdx.x & 31;
            const long b0 = b - lane;
            const long nlive = p.batch - b0 < 32 ? p.batch - b0 : 32;
            const double* tile = smem_ + (long)(threadIdx.x - lane) * (nA + nB);
            // 16-byte accesses when every row of the tile and of A / B starts 16-byte aligned (even nA, nB)
            const bool vec2 = Sys::kStatic && nA % 2 == 0 && nB % 2 == 0;
            if (p.A) {
                double* dstA = p.A + b0 * nA;
                if (vec2) {
                    const int hA = nA / 2, hT = (nA + nB) / 2;
                    const double2* t2p = reinterpret_cast<const double2*>(tile);
                    double2* d2p = reinterpret_cast<double2*>(dstA);
                    for (long e = lane; e < nlive * hA; e += 32) d2p[e] = t2p[(e / hA) * hT + e % hA];
                } else {
                    for (long e = lane; e < nlive * nA; e += 32) dstA[e] = tile[(e / nA) * (nA + nB) + e % nA];
                }
            }
            if constexpr (!Sys::kStatic || (Sys::kStatic && (Sys{}.NU() + Sys{}.NK()) > 0)) {
                if (p.B && nB > 0) {
                    const int nBs = nB > 0 ? nB : 1;
                    double* dstB = p.B + b0 * nB;
                    if (vec2) {
                        const int hA = nA / 2, hB = nBs / 2, hT = (nA + nB) / 2;
                        const double2* t2p = reinterpret_cast<const double2*>(tile);
                        double2* d2p = reinterpret_cast<double2*>(dstB);
                        for (long e = lane; e < nlive * hB; e += 32) d2p[e] = t2p[(e / hB) * hT + hA + e % hB];
                    } else {
                        for (long e = lane; e < nlive * nB; e += 32) dstB[e] = tile[(e / nBs) * (nA + nB) + nA + e % nBs];
                    }
                }
            }
            __syncwarp();
        }
    }
}

template <class Sys>
__global__ void __launch_bounds__(128, lb_min<Sys, true>())
lin_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStrided wsp, const LinParams p,
            const typename Sys::Params par) {
    lin_body<Sys, false>(rsys, dblob, blob_bytes, wsp, p, par, VariedArgs{});
}
template <class Sys>
__global__ void __launch_bounds__(128, lb_min<Sys, true>())
lin_varied_kernel(const RtSys rsys, const char* dblob, int blob_bytes, const WsStrided wsp, const LinParams p,
                  const VariedArgs va) {
    lin_body<Sys, true>(rsys, dblob, blob_bytes, wsp, p, typename Sys::Params{}, va);
}

// ---------------------------------------------------------------------------------------------
template <class Sys>
struct Launchers {
    static typename Sys::Params spec_params(const LaunchCfg& c) {
        typename Sys::Params P{};
        if (Sys::kNPAR > 0 && c.spec_params)
            for (int i = 0; i < Sys::kNPAR; ++i) P.v[i] = c.spec_params[i];
        return P;
    }
    static cudaError_t prep(const void* fn, size_t smem) {
        if (smem > 48 * 1024)
            return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        return cudaSuccess;
    }
    // K for plain launches, KV for per-instance parameters
    template <class P, void (*K)(RtSys, const char*, int, WsStrided, P, typename Sys::Params),
              void (*KV)(RtSys, const char*, int, WsStrided, P, VariedArgs)>
    static cudaError_t launch(const LaunchCfg& c, const P& p, const VariedArgs* va) {
        RtSys rs{};
        if (c.sys) rs = *c.sys;
        cudaError_t e = prep(va ? (const void*)KV : (const void*)K, c.smem);
        if (e != cudaSuccess) return e;
        if (va) KV<<<c.grid, c.block, c.smem, c.stream>>>(rs, c.dblob, c.blob_bytes, c.ws, p, *va);
        else K<<<c.grid, c.block, c.smem, c.stream>>>(rs, c.dblob, c.blob_bytes, c.ws, p, spec_params(c));
        return cudaGetLastError();
    }
    static cudaError_t occupancy(int which, bool varied, int block, size_t smem, int* blocks_per_sm, KernelInfo* info) {
        const void* const fn[2][4] = {
            {(const void*)step_kernel<Sys>, (const void*)p2_kernel<Sys>, (const void*)lin_kernel<Sys>,
             (const void*)project_kernel<Sys>},
            {(const void*)step_varied_kernel<Sys>, (const void*)p2_varied_kernel<Sys>, (const void*)lin_varied_kernel<Sys>,
             (const void*)project_varied_kernel<Sys>}};
        return occupancy_of(fn[varied][which], block, smem, blocks_per_sm, info);
    }
    static cudaError_t occupancy_of(const void* fn, int block, size_t smem, int* blocks_per_sm, KernelInfo* info) {
        cudaFuncAttributes a;
        cudaError_t e = cudaFuncGetAttributes(&a, fn);
        if (e != cudaSuccess) return e;
        if (info) {
            info->regs = a.numRegs;
            info->max_threads = a.maxThreadsPerBlock;
            info->static_smem = a.sharedSizeBytes;
            info->local_bytes = a.localSizeBytes;
        }
        e = prep(fn, smem);
        if (e != cudaSuccess) return e;
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, fn, block, smem);
    }
};

#endif  // __CUDACC__
}  // namespace trepb
#include "trepb_d2.cuh"
namespace trepb {
#if defined(__CUDACC__)

template <class Sys>
KernelSet make_kernelset(const char* name, unsigned long long hash, int specialized, int nX, int nU) {
    KernelSet k;
    k.name = name; k.hash = hash; k.specialized = specialized; k.nX = nX; k.nU = nU;
    k.n_params = Sys::kNPAR;
    using L = Launchers<Sys>;
    k.step = &L::template launch<StepParams, step_kernel<Sys>, step_varied_kernel<Sys>>;
    k.p2 = &L::template launch<P2Params, p2_kernel<Sys>, p2_varied_kernel<Sys>>;
    k.lin = &L::template launch<LinParams, lin_kernel<Sys>, lin_varied_kernel<Sys>>;
    k.proj = &L::template launch<ProjParams, project_kernel<Sys>, project_varied_kernel<Sys>>;
    k.occupancy = &L::occupancy;
    k.d2 = &LaunchersD2<Sys>::run;
    k.d2_occupancy = &LaunchersD2<Sys>::occupancy;
    return k;
}
#endif  // __CUDACC__

}  // namespace trepb
