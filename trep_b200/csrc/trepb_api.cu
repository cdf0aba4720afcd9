// C ABI of libtrepb.so (include/trepb.h): system handles, launch geometry, host<->device staging.
// No CPU fallback: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>
#include "trepb_nvtx.h"
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/trepb.h"
#include "trepb_codegen.h"
#include "trepb_err.h"
#include "trepb_kernels.cuh"
#include "trepb_d2jac.cuh"
#include "trepb_coop.h"
#include "trepb_pack.h"

using namespace trepb;

namespace {
int fail(int code, const std::string& m) { last_error() = m; return code; }
int cuda_fail(cudaError_t e, const char* what) {
    last_error() = std::string(what) + ": " + cudaGetErrorString(e);
    return TREPB_ERR_CUDA;
}
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_fail(e_, #call); } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// dynamic shared memory of a cooperative launch: the description blob, rounded up to an even number of doubles,
// then `teams` workspaces of lay.total doubles
size_t coop_smem(int blob_bytes, int teams, const trepb::CoopLayout& lay) {
    return (size_t)(((blob_bytes + 7) / 8 + 1) & ~1) * 8 + (size_t)teams * lay.total * 8;
}

// Second derivatives by the per-parameter scheme on the tables (trepb_d2jac.cuh) instead of the per-pair kernel of
// `ks`: always for table-driven kernels; for a specialised per-pair kernel whose hyper-dual workspace is far beyond
// the register file (info: its plain d2_kernel).  Measured (evaluations/s, per-pair vs per-parameter): 5-link
// pendulum (31 KB of local memory per thread) 8.1e6 vs 1.1e7, wrench arm (19 KB) 7.8e6 vs 1.2e7; dual pendulums
// (12 KB) 1.05e8 vs 6.8e7, pend-on-cart (10 KB) 1.0e8 vs 6.2e7
bool d2_prefers_jac(const trepb::KernelSet* ks, const trepb::KernelInfo& info) {
    return !ks->specialized || info.local_bytes > 16384;
}
}  // namespace

#if defined(TREPB_PHASE_TIMING)
namespace trepb { __device__ unsigned long long g_phase_ticks[32]; }
extern "C" int trepb_phase_ticks(unsigned long long* out, int reset) {
    cudaError_t e = cudaMemcpyFromSymbol(out, trepb::g_phase_ticks, sizeof(unsigned long long) * 32);
    if (e != cudaSuccess) return TREPB_ERR_CUDA;
    if (reset) {
        unsigned long long z[32] = {0};
        cudaMemcpyToSymbol(trepb::g_phase_ticks, z, sizeof(z));
    }
    return TREPB_OK;
}
#endif

namespace trepb {
SpecRegistry& spec_registry() {
    static SpecRegistry r = {{nullptr}, 0};
    return r;
}
bool spec_register(const KernelSet* ks, unsigned abi) {
    SpecRegistry& r = spec_registry();
    if (abi != kSpecAbi || r.n >= SpecRegistry::kMax) return false;
    r.sets[r.n++] = ks;
    return true;
}
// the first registered kernel set for `hash` that takes n_params run-time parameters, or null
static const KernelSet* spec_find(unsigned long long hash, int n_params) {
    const SpecRegistry& r = spec_registry();
    for (int i = 0; i < r.n; ++i)
        if (r.sets[i]->hash == hash && r.sets[i]->n_params == n_params) return r.sets[i];
    return nullptr;
}
}  // namespace trepb

struct trepb_system {
    int device = 0;
    PackedSys P;
    RtSys dview;            // RtSys whose pointers are device addresses
    char* dblob = nullptr;
    int blob_bytes = 0;
    const KernelSet* ks = nullptr;
    std::vector<double> spec_params;   // run-time parameters of the specialised kernels (param_map order)
    int sms = 0;
    int block = 128;
    int bps[4] = {1, 1, 1, 1};   // resident CTAs per SM for step / p2 / lin / project
    size_t lin_stage_bytes = 0;  // dynamic smem of the staged linearize kernel (0: no staging)
    int lin_bps_staged = 1;
    // team-cooperative path (one warp per instance, workspace in shared memory)
    bool coop = false;
    CoopPack CP;
    char* dcoop = nullptr;
    CoopSys cview;               // base = dcoop
    CoopLayout clay;             // linearize kernel
    CoopLayout clay_solve;       // step / project / p2 kernels (CoopLayout::make, solve_only): smaller, more instances per SM
    int coop_warps_solve = 0;
    int coop_blob_bytes = 0;
    int coop_warps = 0;          // instances in flight per CTA (= per SM)
    const CoopKernelSet* cks = nullptr;
    // general path workspace
    WsStrided wsl;               // layout (base filled per launch)
    int ws_doubles = 0;
    DevBuf ws;
    // second-derivative path: hyper-dual workspace slab + deriv1 scratch (raw arrays, aux, q2, lambda)
    WsStridedT<HDG> wsl_hd;
    int ws_hd_elems = 0;
    DevBuf ws_hd;
    DevBuf d2s[12];
    int bps_d2 = 1;
    // O(nx) second-derivative path (trepb_d2jac.cuh): dual workspace slab + Jacobian-table records
    int flags = 0;
    WsStridedT<Dual> wsl_du;
    int ws_du_elems = 0;
    int bps_d2jac = 1;
    bool d2jac_ok = false;       // pass B's per-CTA working set fits in shared memory for this shape
    bool d2_use_jac = false;     // second derivatives by the per-parameter scheme (trepb_d2jac.cuh)
    DevBuf ws_du, d2g;
    DevBuf coop_ext;             // external slabs of the cooperative linearize kernel (ext flavours)
    // staging for the host-pointer entry points
    DevBuf hb[72];
    cudaStream_t hs[2] = {nullptr, nullptr};   // the two streams the chunked host-pointer calls alternate between
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    // Scratch owned by the handle (the workspace slab of the table-driven thread kernels, the
    // second-derivative scratch) is shared by every launch: a launch that uses it waits, on the device,
    // for the previous such launch - whatever stream that one went to (ScratchGuard).
    cudaEvent_t ev_scratch = nullptr;
    bool scratch_busy = false;
    // per-instance parameters (trepb_*_varied_batch*): the run-time-parameter kernel set of this structure (the
    // handle's own, or the one an all-literal handle was matched against), its occupancy, the map and the table-driven
    // kernels' expanded slots (handle scratch)
    const KernelSet* vks = nullptr;
    bool vinit = false;
    int vbps[4] = {1, 1, 1, 1};
    int vlin_bps_staged = 0;
    bool vd2_use_jac = false;    // second derivatives on vks: as d2_use_jac for a handle built on vks
    int vbps_d2 = 1, vbps_d2jac = 1;
    // vmap_tab: the table-driven layout of the map, for pass A of the per-parameter scheme on a specialised handle
    DevBuf vmap, vmap_tab, vslots;
    // ... on a cooperative handle with TREPB_FLAG_COOP_VARIED: the plan of the link tables' numeric entries and one
    // slot per team of the persistent grid (CoopVaried), allocated at the first varied call
    DevBuf cplan, cvscratch;
    std::mutex mu;       // serialises launches on this handle
    std::mutex mu_host;  // serialises the host-pointer entry points (they share staging buffers)
};

extern "C" {

int trepb_abi_version(void) { return TREPB_ABI_VERSION; }
const char* trepb_last_error(void) { return last_error().c_str(); }

int trepb_device_count(int* n) {
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) { *n = 0; return cuda_fail(e, "cudaGetDeviceCount"); }
    *n = c;
    return TREPB_OK;
}

int trepb_num_specialized(void) { return spec_registry().n; }
const char* trepb_specialized_name(int i) {
    SpecRegistry& r = spec_registry();
    return (i >= 0 && i < r.n) ? r.sets[i]->name : nullptr;
}

// A plug-in is a shared library made of generated specialisation units (trep_b200/build.py: build_plugin):
// loading it runs their static registrars, which add the kernel sets to this library's registries, so that
// trepb_system_create finds a register-resident kernel for a user's own system structure without the library
// being rebuilt.  The plug-in stays loaded for the life of the process (the registries point into it).
int trepb_load_plugin(const char* path, int* n_added) {
    if (n_added) *n_added = 0;
    if (!path) return fail(TREPB_ERR_INVALID, "null path");
    const int before = spec_registry().n + coop_registry().n;
    void* h = dlopen(path, RTLD_NOW | RTLD_LOCAL);
    if (!h) {
        const char* why = dlerror();
        return fail(TREPB_ERR_INVALID, std::string("cannot load plug-in: ") + (why ? why : path));
    }
    const int added = spec_registry().n + coop_registry().n - before;
    if (added <= 0) return fail(TREPB_ERR_INVALID, "the library registered no kernel set (not a trepb plug-in, loaded before, built against other headers than this library, or the registry is full)");
    if (n_added) *n_added = added;
    return TREPB_OK;
}

int trepb_system_create(const trepb_sysdesc* desc, int device, int flags, trepb_system** out) {
    TREPB_NVTX("trepb_system_create");
    if (!out) return fail(TREPB_ERR_INVALID, "null output handle");
    *out = nullptr;
    trepb_system* s = new trepb_system();
    std::string err;
    if (!pack_system(desc, &s->P, &err)) { delete s; return fail(TREPB_ERR_INVALID, err); }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        delete s;
        return fail(TREPB_ERR_CUDA, std::string("no CUDA device (there is no CPU fallback): ") +
                                        (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    }
    if (device < 0 || device >= ndev) { delete s; return fail(TREPB_ERR_INVALID, "device index out of range"); }
    s->device = device;
    s->flags = flags;
#define CUS(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { int rc_ = cuda_fail(e_, #call); trepb_system_destroy(s); return rc_; } } while (0)
    CUS(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUS(cudaGetDeviceProperties(&prop, device));
    s->sms = prop.multiProcessorCount;
    s->blob_bytes = (int)((s->P.blob.size() + 15) & ~size_t(15));
    CUS(cudaMalloc((void**)&s->dblob, s->blob_bytes));
    CUS(cudaMemset(s->dblob, 0, s->blob_bytes));
    CUS(cudaMemcpy(s->dblob, s->P.blob.data(), s->P.blob.size(), cudaMemcpyHostToDevice));
    s->dview = s->P.view(s->dblob);
    // kernel selection
    s->ks = general_kernels();
    ParamMap pm = param_map(s->P);
    const int n_params = (int)pm.values.size();
    if (!(flags & (TREPB_FLAG_NO_SPECIALIZE | TREPB_FLAG_FORCE_COOP))) {
        // an instantiation for exactly this description (every number a literal) if the build made one ...
        const KernelSet* lit = (flags & TREPB_FLAG_NO_LITERAL) ? nullptr : spec_find(desc_hash(s->P), 0);
        if (lit) s->ks = lit;
        // ... else structure picks the kernel and the numbers travel as its run-time parameters
        else if (const KernelSet* ks = spec_find(struct_hash(s->P), n_params)) {
            s->ks = ks;
            s->spec_params = std::move(pm.values);
        }
    }
    s->vks = s->ks;
    // all-literal instantiation: the varied calls run the run-time-parameter kernels of the same structure
    if (s->ks->specialized && s->ks->n_params == 0 && n_params > 0) s->vks = spec_find(struct_hash(s->P), n_params);
    const RtSys& ps = s->P.proto;
    s->ws_doubles = s->wsl.layout(ps.nf, ps.nd, ps.nk, ps.nu, ps.nc);
    // Cooperative kernels for table-driven systems whose per-thread workspace is too large to stay
    // on chip (or when asked for); everything else keeps one thread per instance.
    if (!s->ks->specialized && !(flags & TREPB_FLAG_NO_COOP)) {
        s->CP = coop_pack(desc);
        if (s->CP.ok) {
            CoopSys hv = s->CP.view(s->CP.blob.data());
            const CoopKernelSet* cks = coop_select(hv, !(flags & TREPB_FLAG_NO_SPECIALIZE), (flags & TREPB_FLAG_COOP_ONE_WARP) ? 1 : ((flags & TREPB_FLAG_COOP_TWO_WARPS) ? 2 : 0));
            s->clay.set(hv, cks->specialized != 0, false, cks->ext != 0);
            s->clay_solve.set(hv, cks->specialized != 0, true, cks->ext != 0);
            s->coop_blob_bytes = (int)s->CP.blob.size();
            const size_t blob_d = coop_smem(s->coop_blob_bytes, 0, s->clay);
            const size_t ws_b = (size_t)s->clay.total * 8;
            const size_t cap = (size_t)prop.sharedMemPerBlockOptin;
            int warps = cap > blob_d ? (int)((cap - blob_d) / ws_b) : 0;
            const int lin_cap = cks->max_teams > cks->lin_teams ? cks->max_teams : cks->lin_teams;
            const int solve_cap = cks->max_teams > cks->solve_teams ? cks->max_teams : cks->solve_teams;
            if (warps > lin_cap) warps = lin_cap;
            int warps_solve = cap > blob_d ? (int)((cap - blob_d) / ((size_t)s->clay_solve.total * 8)) : 0;
            if (warps_solve > solve_cap) warps_solve = solve_cap;
            if (const char* e = getenv("TREPB_COOP_WARPS")) {   // diagnostic: fewer instances in flight per SM
                const int w = atoi(e);
                if (w >= 1 && w < warps) warps = w;
                if (w >= 1 && w < warps_solve) warps_solve = w;
            }
            // measured crossover of the table-driven kernels (tools/time_midsize.py, B200): up to ~1000 doubles of thread
            // workspace one thread per instance wins (rod, 656: 1.9x; 5-link pendulum, 955: even), above it the
            // cooperative kernels do (loop3d, 1320: 1.1x linearize / 1.45x step; spring arms, 1461: 1.06x / 1.7x; pccd, 2128: 3.6x / 2.8x)
            const bool wanted = (flags & TREPB_FLAG_FORCE_COOP) || s->ws_doubles > 1200;
            if (warps >= 1 && wanted) {
                CUS(cudaMalloc((void**)&s->dcoop, blob_d));
                CUS(cudaMemset(s->dcoop, 0, blob_d));
                CUS(cudaMemcpy(s->dcoop, s->CP.blob.data(), s->CP.blob.size(), cudaMemcpyHostToDevice));
                s->cview = s->CP.view(s->dcoop);
                s->coop_warps = warps;
                s->coop_warps_solve = warps_solve;
                s->cks = cks;
                s->coop = true;
            }
        }
        if ((flags & TREPB_FLAG_FORCE_COOP) && !s->coop) {
            const std::string why = s->CP.ok ? "workspace does not fit in shared memory" : s->CP.why;
            trepb_system_destroy(s);
            return fail(TREPB_ERR_UNSUPPORTED, "cooperative kernels not available for this system: " + why);
        }
    }
    const size_t base_smem = s->ks->specialized ? 0 : (size_t)s->blob_bytes;
    if (base_smem > 200 * 1024) { trepb_system_destroy(s); return fail(TREPB_ERR_UNSUPPORTED, "system description exceeds shared memory"); }
    for (int w = 0; w < 4; ++w) {
        int b = 0;
        CUS(s->ks->occupancy(w, false, s->block, base_smem, &b, nullptr));
        s->bps[w] = b > 0 ? b : 1;
    }
    s->ws_hd_elems = s->wsl_hd.layout(ps.nf, ps.nd, ps.nk, ps.nu, ps.nc, 1);
    {
        int b = 0;
        KernelInfo ki{};
        CUS(s->ks->d2_occupancy(false, s->block, base_smem, &b, &ki));
        s->bps_d2 = b > 0 ? b : 1;
        s->d2_use_jac = d2_prefers_jac(s->ks, ki);
    }
    // the per-parameter scheme's shape data (also what a per-instance-parameter call on vks may need)
    s->ws_du_elems = s->wsl_du.layout(ps.nf, ps.nd, ps.nk, ps.nu, ps.nc, 2);
    {
        AuxLayout al;
        al.set(ps.nd, ps.nc);
        const int nx = 2 * (ps.nd + ps.nk) + ps.nu;
        s->d2jac_ok = nx <= 1024 && d2solve_smem_needed(ps.nd, ps.nk, ps.nc, nx, al.size) <= (size_t)prop.sharedMemPerBlockOptin;
    }
    if (s->d2_use_jac) {
        int b = 0;
        CUS(d2jac_occupancy(false, s->block, d2jac_smem(s->blob_bytes, s->block, ps.nd, ps.nk), &b, nullptr));
        s->bps_d2jac = b > 0 ? b : 1;
    }
    if (s->ks->specialized) {
        const int nq = ps.nd + ps.nk, nX = 2 * nq, nU = ps.nu + ps.nk;
        const size_t st = (size_t)(nX * nX + nX * nU) * sizeof(double) * s->block;
        if (st <= 160 * 1024) {
            int b = 0;
            CUS(s->ks->occupancy(2, false, s->block, st, &b, nullptr));
            if (b > 0) { s->lin_stage_bytes = st; s->lin_bps_staged = b; }
        }
    }
    CUS(cudaEventCreate(&s->ev0));
    CUS(cudaEventCreate(&s->ev1));
    CUS(cudaEventCreateWithFlags(&s->ev_scratch, cudaEventDisableTiming));
#undef CUS
    *out = s;
    return TREPB_OK;
}

void trepb_system_destroy(trepb_system* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    if (s->dblob) cudaFree(s->dblob);
    if (s->dcoop) cudaFree(s->dcoop);
    s->ws.release();
    s->ws_hd.release();
    s->ws_du.release();
    s->coop_ext.release();
    s->vmap.release();
    s->vmap_tab.release();
    s->vslots.release();
    s->cplan.release();
    s->cvscratch.release();
    s->d2g.release();
    for (auto& b : s->d2s) b.release();
    for (auto& b : s->hb) b.release();
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    if (s->ev_scratch) cudaEventDestroy(s->ev_scratch);
    for (int i = 0; i < 2; ++i) if (s->hs[i]) cudaStreamDestroy(s->hs[i]);
    delete s;
}

int trepb_system_dims(const trepb_system* s, int32_t* nq, int32_t* nd, int32_t* nk, int32_t* nu, int32_t* nc) {
    if (!s) return fail(TREPB_ERR_INVALID, "null system");
    const RtSys& p = s->P.proto;
    if (nq) *nq = p.nd + p.nk;
    if (nd) *nd = p.nd;
    if (nk) *nk = p.nk;
    if (nu) *nu = p.nu;
    if (nc) *nc = p.nc;
    return TREPB_OK;
}

int trepb_system_is_specialized(const trepb_system* s) { return s && s->ks->specialized; }
const char* trepb_system_kernel_name(const trepb_system* s) { return s ? (s->coop ? s->cks->name : s->ks->name) : ""; }
int trepb_system_is_cooperative(const trepb_system* s) { return s && s->coop; }

int trepb_kernel_info(trepb_system* s, int which, int32_t* regs, int32_t* local_bytes, int32_t* blocks_per_sm,
                      int32_t* block, int32_t* smem_bytes) {
    if (!s || which < 0 || which > 3) return fail(TREPB_ERR_INVALID, "bad arguments");
    CU(cudaSetDevice(s->device));
    KernelInfo ki;
    int b = 0;
    if (s->coop) {
        const bool lin = which == 2;
        const int teams = lin ? s->coop_warps : s->coop_warps_solve;
        const bool wide = teams > (lin ? s->cks->lin_teams : s->cks->solve_teams);   // the instantiation a full batch runs
        CU(s->cks->info(which + (wide ? 4 : 0), &ki));
        if (regs) *regs = ki.regs;
        if (local_bytes) *local_bytes = (int32_t)ki.local_bytes;
        if (blocks_per_sm) *blocks_per_sm = 1;
        if (block) *block = 32 * (lin ? s->cks->team_warps : 1) * teams;
        if (smem_bytes) *smem_bytes = (int32_t)coop_smem(s->coop_blob_bytes, teams, lin ? s->clay : s->clay_solve);
        return TREPB_OK;
    }
    size_t smem = s->ks->specialized ? 0 : (size_t)s->blob_bytes;
    if (which == 2 && s->lin_stage_bytes) smem = s->lin_stage_bytes;
    CU(s->ks->occupancy(which, false, s->block, smem, &b, &ki));
    if (regs) *regs = ki.regs;
    if (local_bytes) *local_bytes = (int32_t)ki.local_bytes;
    if (blocks_per_sm) *blocks_per_sm = b;
    if (block) *block = s->block;
    if (smem_bytes) *smem_bytes = (int32_t)smem;
    return TREPB_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------
namespace {

// Grid of a launch whose threads each own a column of a workspace slab of `elem_bytes` x `elems` per thread:
// *grid capped at `resident` CTAs and at ws_grid_cap, and the slab kept within a quarter of the free memory
// (`reclaim`: bytes of handle buffers this launch may reuse, counted as free).  Sizes `slab` to fit.
int slab_grid(long long* grid, long long resident, int elems, size_t elem_bytes, int block, size_t reclaim, DevBuf& slab,
              const char* what) {
    if (*grid > resident) *grid = resident;
    if (*grid > ws_grid_cap(elems, block)) *grid = ws_grid_cap(elems, block);
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    const size_t per_cta = (size_t)elems * elem_bytes * block;
    const size_t budget = (free_b + reclaim) / 4;
    if ((size_t)*grid * per_cta > budget) *grid = (long long)(budget / per_cta);
    if (*grid < 1) return fail(TREPB_ERR_CUDA, std::string("not enough device memory for the ") + what);
    CU(slab.ensure((size_t)*grid * per_cta));
    return TREPB_OK;
}

// grid for `batch` instances at `bps` resident CTAs per SM; for the general path also sizes the
// workspace slab (one column per launched thread).
int make_cfg(trepb_system* s, int which, bool varied, long long batch, int bps, size_t smem, cudaStream_t stream,
             LaunchCfg* c) {
    int block = s->block;
    if (!s->ks->specialized) {
        // small batches of big systems: narrower CTAs so that every SM gets work
        while (block > 32 && (batch + block - 1) / block < 2LL * s->sms) block /= 2;
        if (block != s->block) {
            int b = 0;
            CU((varied ? s->vks : s->ks)->occupancy(which, varied, block, smem, &b, nullptr));
            bps = b > 0 ? b : 1;
        }
    }
    long long grid = (batch + block - 1) / block;
    if (!s->ks->specialized) {
        if (int rc = slab_grid(&grid, (long long)s->sms * bps, s->ws_doubles, sizeof(double), block, s->ws.cap, s->ws,
                               "workspace slab"))
            return rc;
    } else {
        if (grid > 0x7fffffffLL) grid = 0x7fffffffLL;
    }
    if (grid < 1) grid = 1;
    c->grid = (int)grid;
    c->block = block;
    c->smem = smem;
    c->stream = stream;
    c->sys = s->ks->specialized ? nullptr : &s->dview;
    c->dblob = s->dblob;
    c->blob_bytes = s->blob_bytes;
    c->ws = s->wsl;
    c->ws.base = (double*)s->ws.p;
    c->ws.stride = 0;
    c->spec_params = s->spec_params.empty() ? nullptr : s->spec_params.data();
    return TREPB_OK;
}

// persistent grid of the cooperative kernels: one CTA per SM, fewer warps per CTA for small batches
void make_coop(trepb_system* s, long long batch, cudaStream_t stream, CoopLaunch* c, bool solve_only) {
    int warps = solve_only ? s->coop_warps_solve : s->coop_warps;
    const CoopLayout& lay = solve_only ? s->clay_solve : s->clay;
    const long long per_sm = (batch + s->sms - 1) / s->sms;
    if (per_sm < warps) warps = (int)(per_sm < 1 ? 1 : per_sm);
    long long grid = (batch + warps - 1) / warps;
    if (grid > s->sms) grid = s->sms;
    c->grid = (int)grid;
    c->warps = warps;
    c->smem = coop_smem(s->coop_blob_bytes, warps, lay);
    c->stream = stream;
    c->sys = s->cview;
    c->blob_bytes = s->coop_blob_bytes;
    c->lay = lay;
    c->ext = nullptr;
}

// ext flavours of the cooperative kernels: one slab of lay.xtotal doubles per team of the persistent grid
int attach_slabs(trepb_system* s, CoopLaunch* c) {
    if (!c->lay.ext || c->lay.xtotal == 0) return TREPB_OK;
    CU(s->coop_ext.ensure((size_t)c->grid * c->warps * c->lay.xtotal * sizeof(double)));
    c->ext = (double*)s->coop_ext.p;
    return TREPB_OK;
}

// Orders launches that use the handle's scratch across streams: wait for the previous user before the
// launch, mark the end of this one after it.  The caller holds s->mu.
struct ScratchGuard {
    trepb_system* s;
    cudaStream_t st;
    bool on;
    ScratchGuard(trepb_system* s_, cudaStream_t st_, bool on_) : s(s_), st(st_), on(on_) {
        if (on && s->scratch_busy) cudaStreamWaitEvent(st, s->ev_scratch, 0);
    }
    ~ScratchGuard() { if (on) { cudaEventRecord(s->ev_scratch, st); s->scratch_busy = true; } }
};

struct Timed {
    trepb_system* s;
    cudaStream_t st;
    Timed(trepb_system* s_, cudaStream_t st_) : s(s_), st(st_) { cudaEventRecord(s->ev0, st); }
    ~Timed() { cudaEventRecord(s->ev1, st); s->timed = true; }
};

// Uploads the map of a checked `v` (trepb_varied.h) in the specialised (`slots`) or the table-driven layout to `buf`
// and fills va (slots: see varied_slots).
int varied_upload(trepb_system* s, const trepb_varied* v, bool slots, DevBuf& buf_d, cudaStream_t stream, VariedArgs* va) {
    VariedHost H;
    varied_map(s->P, v->n, v->table, v->index, slots, &H);
    // one upload: base, gbase (doubles), then src, gcol (ints)
    const size_t nb = H.base.size(), ng = H.gbase.size();
    std::vector<double> buf(nb + ng + (H.src.size() + H.gcol.size() + 1) / 2 + 1, 0.0);
    memcpy(buf.data(), H.base.data(), nb * sizeof(double));
    if (ng) memcpy(buf.data() + nb, H.gbase.data(), ng * sizeof(double));
    int* ib = (int*)(buf.data() + nb + ng);
    if (!H.src.empty()) memcpy(ib, H.src.data(), H.src.size() * sizeof(int));
    if (!H.gcol.empty()) memcpy(ib + H.src.size(), H.gcol.data(), H.gcol.size() * sizeof(int));
    CU(buf_d.ensure(buf.size() * sizeof(double)));
    // pageable source: returns once the bytes are staged, so `buf` may go out of scope
    CU(cudaMemcpyAsync(buf_d.p, buf.data(), buf.size() * sizeof(double), cudaMemcpyHostToDevice, stream));
    const double* d = (const double*)buf_d.p;
    const int* di = (const int*)(d + nb + ng);
    va->map = H.view(di, d, di + H.src.size(), d + nb);
    va->values = v->values;
    va->slots = nullptr;
    return TREPB_OK;
}

// Per-instance parameters: checks `v` against the handle's description, uploads its map in the layout of vks to
// handle scratch and fills va.  The caller holds s->mu and a ScratchGuard on `stream`.
int varied_setup(trepb_system* s, const trepb_varied* v, cudaStream_t stream, VariedArgs* va) {
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    if (s->coop && !(s->flags & TREPB_FLAG_COOP_VARIED))
        return fail(TREPB_ERR_UNSUPPORTED, "per-instance parameters are not supported by the cooperative kernels (their "
                                           "link tables are built on the host from the description): create the handle "
                                           "with TREPB_FLAG_NO_COOP");
    if (!s->vks) return fail(TREPB_ERR_UNSUPPORTED, "no run-time-parameter kernel set was built for this structure");
    std::string err;
    if (!varied_check(s->P, v->n, v->table, v->index, &err)) return fail(TREPB_ERR_INVALID, err);
    if (v->n > 0 && !v->values) return fail(TREPB_ERR_INVALID, "varied: values is required");
    if (!s->vinit) {
        const size_t smem = s->vks->specialized ? 0 : (size_t)s->blob_bytes;
        for (int w = 0; w < 4; ++w) {
            int b = 0;
            CU(s->vks->occupancy(w, true, s->block, smem, &b, nullptr));
            s->vbps[w] = b > 0 ? b : 1;
        }
        if (s->lin_stage_bytes) CU(s->vks->occupancy(2, true, s->block, s->lin_stage_bytes, &s->vlin_bps_staged, nullptr));
        // second derivatives: the scheme a handle built on vks would pick, and the varied kernels' occupancy
        int b = 0;
        KernelInfo ki{};
        CU(s->vks->d2_occupancy(false, s->block, smem, &b, &ki));
        s->vd2_use_jac = d2_prefers_jac(s->vks, ki);
        CU(s->vks->d2_occupancy(true, s->block, smem, &b, nullptr));
        s->vbps_d2 = b > 0 ? b : 1;
        if (s->vd2_use_jac) {
            const RtSys& ps = s->P.proto;
            CU(d2jac_occupancy(true, s->block, d2jac_smem(s->blob_bytes, s->block, ps.nd, ps.nk), &b, nullptr));
            s->vbps_d2jac = b > 0 ? b : 1;
        }
        s->vinit = true;
    }
    return varied_upload(s, v, s->vks->specialized != 0, s->vmap, stream, va);
}

// table-driven kernels: one expanded parameter vector per launched thread
int varied_slots(trepb_system* s, const LaunchCfg& c, VariedArgs* va) {
    if (s->vks->specialized) return TREPB_OK;
    CU(s->vslots.ensure((size_t)c.grid * c.block * va->map.n_out * sizeof(double)));
    va->slots = (double*)s->vslots.p;
    return TREPB_OK;
}

// Varied cooperative launch: the plan on the device (uploaded once) and the teams' slots, sized once for the widest
// persistent grid of the handle.  The caller holds s->mu and a ScratchGuard on `stream`.
int coop_varied_args(trepb_system* s, const VariedArgs& va, cudaStream_t stream, CoopVaried* cv) {
    const CoopPlan& pl = s->CP.plan;
    if (!s->cplan.p) {
        CU(s->cplan.ensure(pl.ints.size() * sizeof(int32_t)));
        CU(cudaMemcpyAsync(s->cplan.p, pl.ints.data(), pl.ints.size() * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
    }
    const long n8 = (s->coop_blob_bytes + 7) / 8;
    cv->per_team = ((n8 + 1) & ~1L) + 12L * pl.nf;
    const int teams = s->coop_warps > s->coop_warps_solve ? s->coop_warps : s->coop_warps_solve;
    CU(s->cvscratch.ensure((size_t)s->sms * teams * cv->per_team * sizeof(double)));
    cv->map = va.map;
    cv->values = va.values;
    cv->plan = pl.view((const int32_t*)s->cplan.p);
    cv->scratch = (double*)s->cvscratch.p;
    return TREPB_OK;
}

// Launches one call (which: 0 step, 1 p2, 2 lin, 3 project) on the kernels `v` and the handle select: the
// cooperative kernels of a cooperative handle (for per-instance parameters only with TREPB_FLAG_COOP_VARIED: their
// varied instantiations, coop_v(cl, cv)), else the run-time-parameter kernels for per-instance parameters, else one
// thread per instance.  thread(ks, cfg, va) and coop(cl) launch the call's kernel.  stage (linearize with
// A or B, else null): set to 1 when the outputs are staged through shared memory.  vset: the map of `v` when the
// caller has set it up already (varied_setup).  The caller holds s->mu.
template <class Thread, class Coop, class CoopV>
int dispatch(trepb_system* s, int which, long long batch, cudaStream_t stream, const trepb_varied* v, int* stage,
             Thread thread, Coop coop, CoopV coop_v, const VariedArgs* vset = nullptr) {
    if (!v && s->coop) {
        CoopLaunch cl;
        make_coop(s, batch, stream, &cl, which != 2);
        ScratchGuard sg(s, stream, cl.lay.ext != 0);   // ext flavours: slabs owned by the handle
        if (int rc = attach_slabs(s, &cl)) return rc;
        Timed t(s, cl.stream);
        CU(coop(cl));
        return TREPB_OK;
    }
    if (v && s->coop && (s->flags & TREPB_FLAG_COOP_VARIED)) {
        CoopLaunch cl;
        make_coop(s, batch, stream, &cl, which != 2);
        ScratchGuard sg(s, stream, true);   // the teams' slots (and ext slabs) are owned by the handle
        VariedArgs va;
        if (vset) va = *vset;
        else if (int rc = varied_setup(s, v, stream, &va)) return rc;
        CoopVaried cv;
        if (int rc = coop_varied_args(s, va, stream, &cv)) return rc;
        if (int rc = attach_slabs(s, &cl)) return rc;
        if (stage) *stage = 0;
        Timed t(s, cl.stream);
        CU(coop_v(cl, cv));
        return TREPB_OK;
    }
    ScratchGuard sg(s, stream, v || !s->ks->specialized);
    VariedArgs va;
    if (v && vset) va = *vset;
    else if (v)
        if (int rc = varied_setup(s, v, stream, &va)) return rc;
    const int bps_staged = v ? s->vlin_bps_staged : s->lin_bps_staged;
    const bool staged = stage && s->lin_stage_bytes > 0 && bps_staged > 0;
    if (stage) *stage = staged ? 1 : 0;
    const size_t smem = s->ks->specialized ? (staged ? s->lin_stage_bytes : 0) : (size_t)s->blob_bytes;
    LaunchCfg c;
    const int bps = staged ? bps_staged : (v ? s->vbps : s->bps)[which];
    if (int rc = make_cfg(s, which, v != nullptr, batch, bps, smem, stream, &c)) return rc;
    // persistent-style grid: the staged kernel loops with a warp-uniform bound
    if (staged && c.grid > (long long)s->sms * bps_staged) c.grid = (int)((long long)s->sms * bps_staged);
    if (v)
        if (int rc = varied_slots(s, c, &va)) return rc;
    Timed t(s, c.stream);
    CU(thread(v ? s->vks : s->ks, c, v ? &va : nullptr));
    return TREPB_OK;
}

int step_launch(trepb_system* s, const trepb_step_args* a, void* stream, const trepb_varied* v) {
    if (!s || !a) return fail(TREPB_ERR_INVALID, "null argument");
    const RtSys& ps = s->P.proto;
    if (a->batch < 0 || a->nsteps < 1) return fail(TREPB_ERR_INVALID, "batch must be >= 0 and nsteps >= 1");
    if (!a->q1 || !a->p1 || !a->q2 || !a->p2 || !a->status) return fail(TREPB_ERR_INVALID, "q1, p1, q2, p2 and status are required");
    if (ps.nk > 0 && !a->k2) return fail(TREPB_ERR_INVALID, "k2 is required for a system with kinematic configs");
    if (!a->times && !(a->dt != 0.0)) return fail(TREPB_ERR_INVALID, "dt must be non-zero");
    if (a->sample_every < 0) return fail(TREPB_ERR_INVALID, "sample_every must be >= 0");
    if (a->batch == 0) return TREPB_OK;
    std::lock_guard<std::mutex> lk(s->mu);
    CU(cudaSetDevice(s->device));
    StepParams p;
    p.batch = a->batch; p.nsteps = a->nsteps; p.max_it = a->max_iterations;
    p.t0 = a->t0; p.dt = a->dt; p.tol = a->tolerance; p.tolT = sqrt_threshold(a->tolerance);
    p.q1 = a->q1; p.p1 = a->p1; p.u1 = ps.nu ? a->u1 : nullptr; p.k2 = a->k2; p.q2g = a->q2_guess;
    p.lamg = ps.nc ? a->lambda_guess : nullptr;
    p.q2 = a->q2; p.p2 = a->p2; p.lam = ps.nc ? a->lambda1 : nullptr; p.iters = a->iters; p.status = a->status;
    p.sample_every = a->sample_every;
    p.nsamples = a->sample_every > 0 ? a->nsteps / a->sample_every : 0;
    p.traj_q = a->traj_q; p.traj_p = a->traj_p;
    p.times = a->times;
    return dispatch(s, 0, a->batch, (cudaStream_t)stream, v, nullptr,
                    [&](const KernelSet* ks, const LaunchCfg& c, const VariedArgs* va) { return ks->step(c, p, va); },
                    [&](const CoopLaunch& cl) { return s->cks->step(cl, p); },
                    [&](const CoopLaunch& cl, const CoopVaried& cv) { return s->cks->step_v(cl, p, cv); });
}

int project_launch(trepb_system* s, const trepb_project_args* a, void* stream, const trepb_varied* v) {
    if (!s || !a) return fail(TREPB_ERR_INVALID, "null argument");
    if (a->batch < 0 || a->nsteps < 1) return fail(TREPB_ERR_INVALID, "batch must be >= 0 and nsteps >= 1");
    if (!a->bX || !a->bU || !a->Kfb || !a->X || !a->U || !a->status)
        return fail(TREPB_ERR_INVALID, "bX, bU, Kfb, X, U and status are required");
    if (!a->times && !(a->dt != 0.0)) return fail(TREPB_ERR_INVALID, "dt must be non-zero");
    const RtSys& ps = s->P.proto;
    if (ps.nu + ps.nk == 0) return fail(TREPB_ERR_INVALID, "the system has no inputs to feed back");
    if (a->batch == 0) return TREPB_OK;
    std::lock_guard<std::mutex> lk(s->mu);
    CU(cudaSetDevice(s->device));
    ProjParams p;
    p.batch = a->batch; p.nsteps = a->nsteps; p.max_it = a->max_iterations;
    p.t0 = a->t0; p.dt = a->dt; p.tol = a->tolerance; p.tolT = sqrt_threshold(a->tolerance);
    p.bX = a->bX; p.bU = a->bU; p.K = a->Kfb; p.k_per_instance = a->k_per_instance; p.use_hint = a->use_hint;
    p.X = a->X; p.U = a->U; p.iters = a->iters; p.status = a->status; p.fail_step = a->fail_step;
    p.times = a->times;
    return dispatch(s, 3, a->batch, (cudaStream_t)stream, v, nullptr,
                    [&](const KernelSet* ks, const LaunchCfg& c, const VariedArgs* va) { return ks->proj(c, p, va); },
                    [&](const CoopLaunch& cl) { return s->cks->proj(cl, p); },
                    [&](const CoopLaunch& cl, const CoopVaried& cv) { return s->cks->proj_v(cl, p, cv); });
}

// calc_p2 / calc_f / discrete_fm2 share one kernel (P2Params::mode); the caller has validated the pointers
int eval_launch(trepb_system* s, const P2Params& p, void* stream, const trepb_varied* v) {
    if (p.batch == 0) return TREPB_OK;
    std::lock_guard<std::mutex> lk(s->mu);
    CU(cudaSetDevice(s->device));
    return dispatch(s, 1, p.batch, (cudaStream_t)stream, v, nullptr,
                    [&](const KernelSet* ks, const LaunchCfg& c, const VariedArgs* va) { return ks->p2(c, p, va); },
                    [&](const CoopLaunch& cl) { return s->cks->p2(cl, p); },
                    [&](const CoopLaunch& cl, const CoopVaried& cv) { return s->cks->p2_v(cl, p, cv); });
}

int calc_p2_dev(trepb_system* s, int64_t batch, double dt, const double* q0, const double* q1, double* pout,
                const trepb_varied* v, void* stream) {
    if (!s || !q0 || !q1 || !pout) return fail(TREPB_ERR_INVALID, "null argument");
    if (batch < 0 || !(dt != 0.0)) return fail(TREPB_ERR_INVALID, "bad batch or dt");
    P2Params p{};
    p.batch = batch; p.dt = dt; p.q0 = q0; p.q1 = q1; p.p = pout; p.mode = 0;
    return eval_launch(s, p, stream, v);
}

int calc_f_dev(trepb_system* s, int64_t batch, double t1, double t2, const double* q1, const double* q2,
               const double* p1, const double* u1, const double* lambda1, double* f, const trepb_varied* v, void* stream) {
    if (!s || !q1 || !q2 || !p1 || !f) return fail(TREPB_ERR_INVALID, "null argument");
    if (batch < 0 || !(t2 - t1 != 0.0)) return fail(TREPB_ERR_INVALID, "bad batch or t2 == t1");
    P2Params p{};
    p.batch = batch; p.dt = t2 - t1; p.q0 = q1; p.q1 = q2; p.p = f; p.mode = 1;
    p.p1 = p1; p.u1 = s->P.proto.nu ? u1 : nullptr; p.lam = s->P.proto.nc ? lambda1 : nullptr;
    return eval_launch(s, p, stream, v);
}

int discrete_fm2_dev(trepb_system* s, int64_t batch, double t1, double t2, const double* q1, const double* q2,
                     const double* u1, double* fm2, const trepb_varied* v, void* stream) {
    if (!s || !q1 || !q2 || !fm2) return fail(TREPB_ERR_INVALID, "null argument");
    if (batch < 0 || !(t2 - t1 != 0.0)) return fail(TREPB_ERR_INVALID, "bad batch or t2 == t1");
    P2Params p{};
    p.batch = batch; p.dt = t2 - t1; p.q0 = q1; p.q1 = q2; p.p = fm2; p.mode = 2;
    p.u1 = s->P.proto.nu ? u1 : nullptr;
    return eval_launch(s, p, stream, v);
}

// validates + launches the linearize kernel; the caller holds s->mu
// argument checks of a linearize call (also run by deriv2 before it sets anything up)
int lin_check(const trepb_system* s, const trepb_lin_args* a) {
    const RtSys& ps = s->P.proto;
    if (a->batch < 0) return fail(TREPB_ERR_INVALID, "batch must be >= 0");
    if (!a->q1 || !a->p1 || !a->status) return fail(TREPB_ERR_INVALID, "q1, p1 and status are required");
    if (ps.nk > 0 && !a->k2) return fail(TREPB_ERR_INVALID, "k2 is required for a system with kinematic configs");
    if (ps.nu > 0 && !a->u1) return fail(TREPB_ERR_INVALID, "u1 is required for a system with inputs");
    if (!a->t2 && !(a->dt_scalar != 0.0)) return fail(TREPB_ERR_INVALID, "dt must be non-zero");
    if (a->traj_len < 0 || a->traj_len == 1 || (a->traj_len > 1 && a->batch % (a->traj_len - 1) != 0))
        return fail(TREPB_ERR_INVALID, "traj_len must be 0 or >= 2 with batch a multiple of traj_len - 1");
    return TREPB_OK;
}

int lin_launch(trepb_system* s, const trepb_lin_args* a, cudaStream_t stream, double* aux, int aux_size,
               const trepb_varied* v = nullptr, const VariedArgs* vset = nullptr) {
    const RtSys& ps = s->P.proto;
    if (int rc = lin_check(s, a)) return rc;
    if (a->batch == 0) return TREPB_OK;
    CU(cudaSetDevice(s->device));
    LinParams p;
    p.batch = a->batch; p.max_it = a->max_iterations; p.tol = a->tolerance; p.tolT = sqrt_threshold(a->tolerance);
    p.t1s = a->t1_scalar; p.dts = a->dt_scalar; p.t1 = a->t1; p.t2 = a->t2;
    p.q1 = a->q1; p.p1 = a->p1; p.u1 = a->u1; p.k2 = a->k2; p.q2g = a->q2_guess;
    p.lamg = ps.nc ? a->lambda_guess : nullptr;
    p.q2 = a->q2; p.p2 = a->p2; p.lam = ps.nc ? a->lambda1 : nullptr; p.iters = a->iters; p.status = a->status;
    p.A = a->A; p.B = (ps.nu + ps.nk) > 0 ? a->B : nullptr;
    double* raw[12] = {a->q2_dq1, a->q2_dp1, a->q2_du1, a->q2_dk2, a->p2_dq1, a->p2_dp1, a->p2_du1, a->p2_dk2,
                       a->l1_dq1, a->l1_dp1, a->l1_du1, a->l1_dk2};
    for (int i = 0; i < 12; ++i) p.raw[i] = raw[i];
    p.aux = aux; p.aux_size = aux_size;
    p.traj_len = a->traj_len;
    p.stage = 0;
    return dispatch(s, 2, a->batch, stream, v, (p.A || p.B) ? &p.stage : nullptr,
                    [&](const KernelSet* ks, const LaunchCfg& c, const VariedArgs* va) { return ks->lin(c, p, va); },
                    [&](const CoopLaunch& cl) {
                        AuxLayout al;
                        al.set(ps.nd, ps.nc);
                        return s->cks->lin(cl, p, al);
                    },
                    [&](const CoopLaunch& cl, const CoopVaried& cv) {
                        AuxLayout al;
                        al.set(ps.nd, ps.nc);
                        return s->cks->lin_v(cl, p, al, cv);
                    }, vset);
}

int lin_dev(trepb_system* s, const trepb_lin_args* a, void* stream, const trepb_varied* v) {
    if (!s || !a) return fail(TREPB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(s->mu);
    return lin_launch(s, a, (cudaStream_t)stream, nullptr, 0, v);
}
}  // namespace

extern "C" {

int trepb_step_batch_dev(trepb_system* s, const trepb_step_args* a, void* stream) {
    TREPB_NVTX("trepb_step_batch_dev");
    return step_launch(s, a, stream, nullptr);
}

int trepb_step_varied_batch_dev(trepb_system* s, const trepb_step_args* a, const trepb_varied* v, void* stream) {
    TREPB_NVTX("trepb_step_varied_batch_dev");
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    return step_launch(s, a, stream, v);
}

int trepb_project_batch_dev(trepb_system* s, const trepb_project_args* a, void* stream) {
    TREPB_NVTX("trepb_project_batch_dev");
    return project_launch(s, a, stream, nullptr);
}

int trepb_project_varied_batch_dev(trepb_system* s, const trepb_project_args* a, const trepb_varied* v, void* stream) {
    TREPB_NVTX("trepb_project_varied_batch_dev");
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    return project_launch(s, a, stream, v);
}

int trepb_calc_p2_batch_dev(trepb_system* s, int64_t batch, double dt, const double* q0, const double* q1,
                            double* pout, void* stream) {
    TREPB_NVTX("trepb_calc_p2_batch_dev");
    return calc_p2_dev(s, batch, dt, q0, q1, pout, nullptr, stream);
}

int trepb_calc_p2_varied_batch_dev(trepb_system* s, int64_t batch, double dt, const double* q0, const double* q1,
                                   double* pout, const trepb_varied* v, void* stream) {
    TREPB_NVTX("trepb_calc_p2_varied_batch_dev");
    if (!v) return fail(TREPB_ERR_INVALID, "null argument");
    return calc_p2_dev(s, batch, dt, q0, q1, pout, v, stream);
}

int trepb_calc_f_batch_dev(trepb_system* s, int64_t batch, double t1, double t2, const double* q1, const double* q2,
                           const double* p1, const double* u1, const double* lambda1, double* f, void* stream) {
    TREPB_NVTX("trepb_calc_f_batch_dev");
    return calc_f_dev(s, batch, t1, t2, q1, q2, p1, u1, lambda1, f, nullptr, stream);
}

int trepb_calc_f_varied_batch_dev(trepb_system* s, int64_t batch, double t1, double t2, const double* q1,
                                  const double* q2, const double* p1, const double* u1, const double* lambda1,
                                  double* f, const trepb_varied* v, void* stream) {
    TREPB_NVTX("trepb_calc_f_varied_batch_dev");
    if (!v) return fail(TREPB_ERR_INVALID, "null argument");
    return calc_f_dev(s, batch, t1, t2, q1, q2, p1, u1, lambda1, f, v, stream);
}

int trepb_discrete_fm2_batch_dev(trepb_system* s, int64_t batch, double t1, double t2, const double* q1,
                                 const double* q2, const double* u1, double* fm2, void* stream) {
    TREPB_NVTX("trepb_discrete_fm2_batch_dev");
    return discrete_fm2_dev(s, batch, t1, t2, q1, q2, u1, fm2, nullptr, stream);
}

int trepb_discrete_fm2_varied_batch_dev(trepb_system* s, int64_t batch, double t1, double t2, const double* q1,
                                        const double* q2, const double* u1, double* fm2, const trepb_varied* v,
                                        void* stream) {
    TREPB_NVTX("trepb_discrete_fm2_varied_batch_dev");
    if (!v) return fail(TREPB_ERR_INVALID, "null argument");
    return discrete_fm2_dev(s, batch, t1, t2, q1, q2, u1, fm2, v, stream);
}

int trepb_varied_check(const trepb_sysdesc* desc, const trepb_varied* v) {
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    PackedSys P;
    std::string err;
    if (!pack_system(desc, &P, &err)) return fail(TREPB_ERR_INVALID, err);
    if (!varied_check(P, v->n, v->table, v->index, &err)) return fail(TREPB_ERR_INVALID, err);
    return TREPB_OK;
}

int trepb_linearize_batch_dev(trepb_system* s, const trepb_lin_args* a, void* stream) {
    TREPB_NVTX("trepb_linearize_batch_dev");
    return lin_dev(s, a, stream, nullptr);
}

int trepb_linearize_varied_batch_dev(trepb_system* s, const trepb_lin_args* a, const trepb_varied* v, void* stream) {
    TREPB_NVTX("trepb_linearize_varied_batch_dev");
    if (!v) return fail(TREPB_ERR_INVALID, "null argument");
    return lin_dev(s, a, stream, v);
}

// deriv1 (the linearize kernel, exporting the factorizations) + second derivatives.  Per-instance parameters (v): one
// row per instance, the map uploaded once (varied_setup) and used by both launches, on the run-time-parameter kernels
// of the structure (vks).  Every launch-geometry and scratch decision is made before the first launch, so that the
// table-driven slots are sized once for both.
static int d2_dev(trepb_system* s, const trepb_d2_args* a, cudaStream_t stream, const trepb_varied* v) {
    if (!s || !a) return fail(TREPB_ERR_INVALID, "null argument");
    const RtSys& ps = s->P.proto;
    const int nd = ps.nd, nk = ps.nk, nq = nd + nk, nu = ps.nu, nc = ps.nc;
    const long long B = a->lin.batch;
    if (B < 0) return fail(TREPB_ERR_INVALID, "batch must be >= 0");
    if (v && a->lin.traj_len != 0)
        return fail(TREPB_ERR_INVALID, "per-instance parameters of second derivatives take one row per instance: "
                                       "traj_len must be 0");
    if (B == 0) return TREPB_OK;
    if (int rc = lin_check(s, &a->lin)) return rc;   // before any scratch, zeroing or launch of this call
    std::lock_guard<std::mutex> lk(s->mu);
    CU(cudaSetDevice(s->device));
    ScratchGuard sg(s, stream, true);   // covers the linearize launch below and both second-derivative passes
    VariedArgs va{};
    const KernelSet* ks = s->ks;
    bool use_jac = s->d2_use_jac;
    if (v) {
        if (int rc = varied_setup(s, v, stream, &va)) return rc;
        ks = s->vks;
        use_jac = s->vd2_use_jac;
    }
    // deriv1 products this kernel consumes: use the caller's arrays where given, scratch otherwise
    trepb_lin_args la = a->lin;
    const size_t cnt[4] = {(size_t)nq, (size_t)nd, (size_t)nu, (size_t)nk};
    double** qd[4] = {&la.q2_dq1, &la.q2_dp1, &la.q2_du1, &la.q2_dk2};
    double** ld[4] = {&la.l1_dq1, &la.l1_dp1, &la.l1_du1, &la.l1_dk2};
    int k = 0;
    for (int i = 0; i < 4; ++i) {
        if (!*qd[i]) { CU(s->d2s[k].ensure((size_t)B * cnt[i] * nd * sizeof(double) + 8)); *qd[i] = (double*)s->d2s[k].p; }
        ++k;
        if (!*ld[i]) { CU(s->d2s[k].ensure((size_t)B * cnt[i] * nc * sizeof(double) + 8)); *ld[i] = (double*)s->d2s[k].p; }
        ++k;
    }
    if (!la.q2) { CU(s->d2s[k].ensure((size_t)B * nq * sizeof(double))); la.q2 = (double*)s->d2s[k].p; }
    ++k;
    if (nc && !la.lambda1) { CU(s->d2s[k].ensure((size_t)B * nc * sizeof(double))); la.lambda1 = (double*)s->d2s[k].p; }
    ++k;
    AuxLayout al;
    al.set(nd, nc);
    CU(s->d2s[k].ensure((size_t)B * al.size * sizeof(double)));
    double* aux = (double*)s->d2s[k].p;
    D2Params p;
    p.batch = B;
    p.nx = nq + nd + nu + nk;
    p.npairs = p.nx * (p.nx + 1) / 2;
    p.t1s = la.t1_scalar; p.dts = la.dt_scalar; p.t1 = la.t1; p.t2 = la.t2;
    p.q1 = la.q1; p.u1 = la.u1; p.q2 = la.q2; p.lam = la.lambda1;
    for (int i = 0; i < 4; ++i) { p.q2_d[i] = *qd[i]; p.l1_d[i] = *ld[i]; }
    p.aux = aux; p.auxl = al; p.status = la.status;
    for (int w = 0; w < 3; ++w)
        for (int kd = 0; kd < 10; ++kd) p.out[w][kd] = a->d2[10 * w + kd];
    if (nc == 0) for (int kd = 0; kd < 10; ++kd) p.out[2][kd] = nullptr;
    {
        const size_t nX = 2 * (size_t)nq, nU = (size_t)(nu + nk);
        p.z = a->z; p.zxx = a->z ? a->fdxdx : nullptr; p.zxu = a->z ? a->fdxdu : nullptr; p.zuu = a->z ? a->fdudu : nullptr;
        if (p.zxx) CU(cudaMemsetAsync(p.zxx, 0, (size_t)B * nX * nX * sizeof(double), stream));
        if (p.zxu && nU) CU(cudaMemsetAsync(p.zxu, 0, (size_t)B * nX * nU * sizeof(double), stream));
        if (p.zuu && nU) CU(cudaMemsetAsync(p.zuu, 0, (size_t)B * nU * nU * sizeof(double), stream));
        if (nU == 0) { p.zxu = nullptr; p.zuu = nullptr; }
    }
    // ---- launch geometry of the second-derivative pass(es)
    const bool jac = use_jac && !(s->flags & TREPB_FLAG_D2_PAIRWISE) && s->d2jac_ok;
    LaunchCfg c;
    c.ws = s->wsl;
    c.dblob = s->dblob; c.blob_bytes = s->blob_bytes; c.stream = stream;
    c.block = s->block;
    // per-instance parameters of pass A / of the per-pair kernel: the map of the linearize launch, except on a
    // specialised handle that takes the per-parameter scheme (pass A is table-driven there: its own map layout)
    VariedArgs vd = va;
    long long d2_threads = 0;   // threads that need a table-driven slot
    JacLayout jl;
    long long nb = 0, jgrid = 0;
    WsStridedT<Dual> wd = s->wsl_du;
    WsStridedT<HDG> w = s->wsl_hd;
    if (jac) {
        // pass A: one dual evaluation of the Jacobian tables per (instance, parameter);
        // pass B: contraction + solves per pair (trepb_d2jac.cuh).  The batch is processed in
        // chunks so that the table records stay within a few GB.
        jl.set(nd, nk, nu, nc);
        size_t free_b = 0, total_b = 0;
        CU(cudaMemGetInfo(&free_b, &total_b));
        const size_t avail = free_b + s->ws_du.cap + s->d2g.cap;
        const size_t per_inst = (size_t)p.nx * jl.size * sizeof(double);
        size_t gbudget = avail / 4;
        if (gbudget > ((size_t)4 << 30)) gbudget = (size_t)4 << 30;
        nb = (long long)(gbudget / per_inst);
        if (nb < 1) return fail(TREPB_ERR_CUDA, "not enough device memory for the second-derivative table records");
        if (nb > B) nb = B;
        jgrid = (nb * p.nx + c.block - 1) / c.block;
        if (int rc = slab_grid(&jgrid, (long long)s->sms * (v ? s->vbps_d2jac : s->bps_d2jac), s->ws_du_elems, sizeof(Dual),
                               c.block, s->ws_du.cap + s->d2g.cap, s->ws_du, "second-derivative workspace"))
            return rc;
        CU(s->d2g.ensure((size_t)nb * per_inst));
        wd.base = (Dual*)s->ws_du.p; wd.stride = 0;
        c.spec_params = nullptr;
        c.smem = d2jac_smem(s->blob_bytes, c.block, nd, nk);
        c.sys = &s->dview;
        if (v && ks->specialized)
            if (int rc = varied_upload(s, v, false, s->vmap_tab, stream, &vd)) return rc;
        if (v) d2_threads = jgrid * c.block;
    } else {
        // one thread per (instance, parameter s, block of kD2Dirs directions t)
        const long long threads = B * (long long)d2_blocks(p.nx, ks->specialized ? 1 : kD2Dirs);
        long long grid = (threads + c.block - 1) / c.block;
        w.base = nullptr; w.stride = 0;
        if (!ks->specialized) {
            if (int rc = slab_grid(&grid, (long long)s->sms * (v ? s->vbps_d2 : s->bps_d2), s->ws_hd_elems, sizeof(HDG),
                                   c.block, s->ws_hd.cap, s->ws_hd, "second-derivative workspace"))
                return rc;
            w.base = (HDG*)s->ws_hd.p;
            if (v) d2_threads = grid * c.block;
        } else if (grid > 0x7fffffffLL) grid = 0x7fffffffLL;
        c.spec_params = s->spec_params.empty() ? nullptr : s->spec_params.data();
        c.grid = (int)grid;
        c.smem = ks->specialized ? 0 : (size_t)s->blob_bytes;
        c.sys = ks->specialized ? nullptr : &s->dview;
    }
    // table-driven slots for the larger of the two launches: this call's linearize launch may still grow vslots
    // (varied_slots) before it runs, never between it and the launches below
    if (d2_threads) CU(s->vslots.ensure((size_t)d2_threads * vd.map.n_out * sizeof(double)));
    if (int rc = lin_launch(s, &la, stream, aux, al.size, v, v ? &va : nullptr)) return rc;
    if (d2_threads) vd.slots = (double*)s->vslots.p;
    const VariedArgs* vp = v ? &vd : nullptr;
    Timed t(s, stream);
    if (jac) {
        for (long long b0 = 0; b0 < B; b0 += nb) {
            const long long cnt_b = B - b0 < nb ? B - b0 : nb;
            long long g = (cnt_b * p.nx + c.block - 1) / c.block;
            c.grid = (int)(g < jgrid ? g : jgrid);
            CU(d2jac_run(c, wd, p, (double*)s->d2g.p, jl, (long)b0, (long)cnt_b, vp));
            // pass B reads deriv1's factors, the table records and the tangents, not the system: no varied flavour
            CU(d2solve_run(stream, p, (const double*)s->d2g.p, jl, nd, nk, nu, nc, (long)b0, (long)cnt_b));
        }
        return TREPB_OK;
    }
    CU(ks->d2(c, w, p, vp));
    return TREPB_OK;
}

int trepb_deriv2_batch_dev(trepb_system* s, const trepb_d2_args* a, void* stream) {
    TREPB_NVTX("trepb_deriv2_batch_dev");
    return d2_dev(s, a, (cudaStream_t)stream, nullptr);
}

int trepb_deriv2_varied_batch_dev(trepb_system* s, const trepb_d2_args* a, const trepb_varied* v, void* stream) {
    TREPB_NVTX("trepb_deriv2_varied_batch_dev");
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    return d2_dev(s, a, (cudaStream_t)stream, v);
}

int trepb_last_kernel_ms(trepb_system* s, float* ms) {
    if (!s || !ms) return fail(TREPB_ERR_INVALID, "null argument");
    if (!s->timed) return fail(TREPB_ERR_INVALID, "no kernel has been launched on this system");
    CU(cudaSetDevice(s->device));
    CU(cudaEventSynchronize(s->ev1));
    CU(cudaEventElapsedTime(ms, s->ev0, s->ev1));
    return TREPB_OK;
}

// ---- device utilities -------------------------------------------------------------------------
int trepb_malloc(int device, int64_t bytes, void** ptr) {
    CU(cudaSetDevice(device));
    CU(cudaMalloc(ptr, (size_t)(bytes > 0 ? bytes : 1)));
    return TREPB_OK;
}
int trepb_free(int device, void* ptr) {
    CU(cudaSetDevice(device));
    CU(cudaFree(ptr));
    return TREPB_OK;
}
int trepb_host_alloc(int64_t bytes, void** ptr) {
    CU(cudaHostAlloc(ptr, (size_t)(bytes > 0 ? bytes : 1), cudaHostAllocDefault));
    return TREPB_OK;
}
int trepb_host_free(void* ptr) {
    CU(cudaFreeHost(ptr));
    return TREPB_OK;
}
int trepb_memcpy_h2d(int device, void* dst, const void* src, int64_t bytes) {
    CU(cudaSetDevice(device));
    CU(cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyHostToDevice));
    return TREPB_OK;
}
int trepb_memcpy_d2h(int device, void* dst, const void* src, int64_t bytes) {
    CU(cudaSetDevice(device));
    CU(cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost));
    return TREPB_OK;
}
int trepb_memcpy_d2d(int device, void* dst, const void* src, int64_t bytes) {
    CU(cudaSetDevice(device));
    CU(cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyDeviceToDevice));
    return TREPB_OK;
}
int trepb_memset(int device, void* dst, int value, int64_t bytes) {
    CU(cudaSetDevice(device));
    CU(cudaMemset(dst, value, (size_t)bytes));
    return TREPB_OK;
}
int trepb_synchronize(int device) {
    CU(cudaSetDevice(device));
    CU(cudaDeviceSynchronize());
    return TREPB_OK;
}

// ---- host-pointer entry points: copy in, run, copy out, synchronize ---------------------------
}  // extern "C"

namespace {
struct Stager {
    trepb_system* s;
    int k = 0;
    struct Out { void* host; void* dev; size_t bytes; } outs[72];
    int nout = 0;
    int err = 0;
    explicit Stager(trepb_system* s_) : s(s_) {}
    template <class T>
    const T* in(const T* host, size_t count) {
        if (!host || err) return nullptr;
        DevBuf& b = s->hb[k++];
        const size_t bytes = count * sizeof(T);
        cudaError_t e = b.ensure(bytes ? bytes : 8);
        if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(b.p, host, bytes, cudaMemcpyHostToDevice, 0);
        if (e != cudaSuccess) { err = cuda_fail(e, "staging host input"); return nullptr; }
        return (const T*)b.p;
    }
    template <class T>
    T* out(T* host, size_t count) {
        if (!host || err) return nullptr;
        DevBuf& b = s->hb[k++];
        const size_t bytes = count * sizeof(T);
        cudaError_t e = b.ensure(bytes ? bytes : 8);
        // the staging buffers are reused between calls: clear, so that what a kernel does not write (the rows
        // after a failed step of a rollout) reads as zeros, not as an earlier call's data
        if (e == cudaSuccess && bytes) e = cudaMemsetAsync(b.p, 0, bytes, 0);
        if (e != cudaSuccess) { err = cuda_fail(e, "staging host output"); return nullptr; }
        outs[nout++] = {host, b.p, bytes};
        return (T*)b.p;
    }
    // per-instance parameters: `rows` rows of v->n values
    trepb_varied dv{};
    const trepb_varied* varied(const trepb_varied* v, size_t rows) {
        if (!v) return nullptr;
        dv = *v;
        dv.values = in(v->values, rows * v->n);
        return &dv;
    }
    int finish() {
        for (int i = 0; i < nout; ++i)
            if (outs[i].bytes) CU(cudaMemcpyAsync(outs[i].host, outs[i].dev, outs[i].bytes, cudaMemcpyDeviceToHost, 0));
        CU(cudaStreamSynchronize(0));
        return TREPB_OK;
    }
};
// Chunked variant for large batches: the batch is cut into a few contiguous chunks that alternate between two
// streams - host-to-device copy, kernel and device-to-host copy of a chunk are ordered on its stream, so the
// copies of one chunk overlap the kernel of another (and each other: the two directions use different copy
// engines).  Every per-instance array is registered with its element count per instance; chunk c covers the
// instances [lo, lo + n).  Host buffers should be pinned for the copies to be asynchronous.
struct Pipe {
    trepb_system* s;
    size_t B;
    struct Arr { const char* hin; char* hout; char* dev; size_t per; } arr[40];
    int n = 0, k = 0, err = 0;
    Pipe(trepb_system* s_, size_t B_) : s(s_), B(B_) {}
    char* reg(const void* hin, void* hout, size_t per_bytes) {
        if (err) return nullptr;
        DevBuf& b = s->hb[k++];
        cudaError_t e = b.ensure(B * per_bytes ? B * per_bytes : 8);
        if (e != cudaSuccess) { err = cuda_fail(e, "staging buffers"); return nullptr; }
        arr[n++] = {(const char*)hin, (char*)hout, (char*)b.p, per_bytes};
        return (char*)b.p;
    }
    static constexpr bool kIn = true, kOut = false;
    template <class T> void field(T*& p, size_t per, bool input) {
        if (p) p = (T*)reg(input ? (const void*)p : nullptr, input ? nullptr : (void*)p, per * sizeof(T));
    }
    static int chunks(size_t B) { return B >= 4 * 65536 ? 4 : (B >= 2 * 65536 ? 2 : 1); }
    int streams() {
        for (int i = 0; i < 2; ++i)
            if (!s->hs[i]) CU(cudaStreamCreateWithFlags(&s->hs[i], cudaStreamNonBlocking));
        return TREPB_OK;
    }
    int upload(size_t lo, size_t cnt, cudaStream_t st) {
        for (int i = 0; i < n; ++i) {
            const size_t off = lo * arr[i].per, bytes = cnt * arr[i].per;
            if (!bytes) continue;
            if (arr[i].hin) CU(cudaMemcpyAsync(arr[i].dev + off, arr[i].hin + off, bytes, cudaMemcpyHostToDevice, st));
            else CU(cudaMemsetAsync(arr[i].dev + off, 0, bytes, st));   // see Stager::out
        }
        return TREPB_OK;
    }
    int download(size_t lo, size_t cnt, cudaStream_t st) {
        for (int i = 0; i < n; ++i) {
            const size_t off = lo * arr[i].per, bytes = cnt * arr[i].per;
            if (arr[i].hout && bytes) CU(cudaMemcpyAsync(arr[i].hout + off, arr[i].dev + off, bytes, cudaMemcpyDeviceToHost, st));
        }
        return TREPB_OK;
    }
    int finish() {
        for (int i = 0; i < 2; ++i) CU(cudaStreamSynchronize(s->hs[i]));
        return TREPB_OK;
    }
    // Runs launch(&args, varied, stream) on C_ chunks.  fields(x, f) calls f(x.member, elements per instance,
    // kIn or kOut) for every per-instance array of x; the parameter rows of v (one per instance) are chunked too.
    template <class Args, class Fields, class Launch>
    int run(Args d, const trepb_varied* v, int C_, Fields fields, Launch launch) {
        fields(d, [&](auto& p, size_t per, bool input) { field(p, per, input); });
        trepb_varied dv{};
        if (v) { dv = *v; field(dv.values, (size_t)v->n, kIn); }
        if (err) return err;
        int rc = streams();
        if (rc) return rc;
        for (int c = 0; c < C_; ++c) {
            const size_t lo = B * c / C_, hi = B * (c + 1) / C_, cnt = hi - lo;
            cudaStream_t st = s->hs[c & 1];
            if ((rc = upload(lo, cnt, st))) return rc;
            Args e = d;
            e.batch = (int64_t)cnt;
            fields(e, [&](auto& p, size_t per, bool) { if (p) p += lo * per; });
            trepb_varied ev = dv;
            if (ev.values) ev.values += lo * (size_t)v->n;
            if ((rc = launch(&e, v ? &ev : nullptr, st))) return rc;
            if ((rc = download(lo, cnt, st))) return rc;
        }
        return finish();
    }
};
}  // namespace

extern "C" {

static int step_host(trepb_system* s, const trepb_step_args* a, const trepb_varied* v) {
    if (!s || !a) return fail(TREPB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> hlk(s->mu_host);
    if (a->batch < 0 || a->nsteps < 1) return fail(TREPB_ERR_INVALID, "batch must be >= 0 and nsteps >= 1");
    const RtSys& ps = s->P.proto;
    const size_t B = (size_t)a->batch, nq = ps.nd + ps.nk, nd = ps.nd, nu = ps.nu, nk = ps.nk, nc = ps.nc, K = (size_t)a->nsteps;
    const size_t ns = a->sample_every > 0 ? (size_t)(a->nsteps / a->sample_every) : 0;
    CU(cudaSetDevice(s->device));
    if (const int C_ = Pipe::chunks(B); C_ > 1 && a->q1 && a->p1 && a->q2 && a->p2 && a->status) {
        Pipe pp(s, B);
        trepb_step_args d = *a;
        if (a->times) {   // shared by every chunk: up before either stream starts
            DevBuf& tb = s->hb[pp.k++];
            CU(tb.ensure((K + 1) * sizeof(double)));
            CU(cudaMemcpy(tb.p, a->times, (K + 1) * sizeof(double), cudaMemcpyHostToDevice));
            d.times = (const double*)tb.p;
        }
        constexpr bool kIn = Pipe::kIn, kOut = Pipe::kOut;
        return pp.run(d, v, C_, [&](trepb_step_args& x, auto&& f) {
            f(x.q1, nq, kIn); f(x.p1, nd, kIn); f(x.u1, K * nu, kIn); f(x.k2, K * nk, kIn);
            f(x.q2_guess, nd, kIn); f(x.lambda_guess, nc, kIn);
            f(x.q2, nq, kOut); f(x.p2, nd, kOut); f(x.lambda1, nc, kOut); f(x.iters, 1, kOut); f(x.status, 1, kOut);
            f(x.traj_q, ns * nq, kOut); f(x.traj_p, ns * nd, kOut);
        }, [&](const trepb_step_args* e, const trepb_varied* ev, cudaStream_t st) { return step_launch(s, e, st, ev); });
    }
    Stager st(s);
    trepb_step_args d = *a;
    d.q1 = st.in(a->q1, B * nq); d.p1 = st.in(a->p1, B * nd);
    d.u1 = st.in(a->u1, B * K * nu); d.k2 = st.in(a->k2, B * K * nk);
    d.q2_guess = st.in(a->q2_guess, B * nd); d.lambda_guess = st.in(a->lambda_guess, B * nc);
    d.q2 = st.out(a->q2, B * nq); d.p2 = st.out(a->p2, B * nd); d.lambda1 = st.out(a->lambda1, B * nc);
    d.iters = st.out(a->iters, B); d.status = st.out(a->status, B);
    d.traj_q = st.out(a->traj_q, B * ns * nq); d.traj_p = st.out(a->traj_p, B * ns * nd);
    d.times = st.in(a->times, K + 1);
    const trepb_varied* dv = st.varied(v, B);
    if (st.err) return st.err;
    int rc = step_launch(s, &d, nullptr, dv);
    if (rc) return rc;
    return st.finish();
}

int trepb_step_batch(trepb_system* s, const trepb_step_args* a) {
    TREPB_NVTX("trepb_step_batch");
    return step_host(s, a, nullptr);
}

int trepb_step_varied_batch(trepb_system* s, const trepb_step_args* a, const trepb_varied* v) {
    TREPB_NVTX("trepb_step_varied_batch");
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    return step_host(s, a, v);
}

static int project_host(trepb_system* s, const trepb_project_args* a, const trepb_varied* v) {
    if (!s || !a) return fail(TREPB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> hlk(s->mu_host);
    if (a->batch < 0 || a->nsteps < 1) return fail(TREPB_ERR_INVALID, "batch must be >= 0 and nsteps >= 1");
    const RtSys& ps = s->P.proto;
    const size_t B = (size_t)a->batch, K = (size_t)a->nsteps, nX = 2 * (size_t)(ps.nd + ps.nk), nU = (size_t)(ps.nu + ps.nk);
    CU(cudaSetDevice(s->device));
    Stager st(s);
    trepb_project_args d = *a;
    d.bX = st.in(a->bX, B * (K + 1) * nX); d.bU = st.in(a->bU, B * K * nU);
    d.Kfb = st.in(a->Kfb, (a->k_per_instance ? B : 1) * K * nU * nX);
    d.X = st.out(a->X, B * (K + 1) * nX); d.U = st.out(a->U, B * K * nU);
    d.iters = st.out(a->iters, B); d.status = st.out(a->status, B); d.fail_step = st.out(a->fail_step, B);
    d.times = st.in(a->times, K + 1);
    const trepb_varied* dv = st.varied(v, B);
    if (st.err) return st.err;
    int rc = project_launch(s, &d, nullptr, dv);
    if (rc) return rc;
    return st.finish();
}

int trepb_project_batch(trepb_system* s, const trepb_project_args* a) {
    TREPB_NVTX("trepb_project_batch");
    return project_host(s, a, nullptr);
}

int trepb_project_varied_batch(trepb_system* s, const trepb_project_args* a, const trepb_varied* v) {
    TREPB_NVTX("trepb_project_varied_batch");
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    return project_host(s, a, v);
}

static int calc_p2_host(trepb_system* s, int64_t batch, double dt, const double* q0, const double* q1, double* p,
                        const trepb_varied* v) {
    if (!s) return fail(TREPB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> hlk(s->mu_host);
    if (batch < 0) return fail(TREPB_ERR_INVALID, "batch must be >= 0");
    const RtSys& ps = s->P.proto;
    const size_t B = (size_t)batch, nq = ps.nd + ps.nk;
    CU(cudaSetDevice(s->device));
    Stager st(s);
    const double* dq0 = st.in(q0, B * nq);
    const double* dq1 = st.in(q1, B * nq);
    double* dp = st.out(p, B * ps.nd);
    const trepb_varied* dv = st.varied(v, B);
    if (st.err) return st.err;
    int rc = calc_p2_dev(s, batch, dt, dq0, dq1, dp, dv, nullptr);
    if (rc) return rc;
    return st.finish();
}

int trepb_calc_p2_batch(trepb_system* s, int64_t batch, double dt, const double* q0, const double* q1, double* p) {
    TREPB_NVTX("trepb_calc_p2_batch");
    return calc_p2_host(s, batch, dt, q0, q1, p, nullptr);
}

int trepb_calc_p2_varied_batch(trepb_system* s, int64_t batch, double dt, const double* q0, const double* q1,
                               double* p, const trepb_varied* v) {
    TREPB_NVTX("trepb_calc_p2_varied_batch");
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    return calc_p2_host(s, batch, dt, q0, q1, p, v);
}

static int calc_f_host(trepb_system* s, int64_t batch, double t1, double t2, const double* q1, const double* q2,
                       const double* p1, const double* u1, const double* lambda1, double* f, const trepb_varied* v) {
    if (!s) return fail(TREPB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> hlk(s->mu_host);
    if (batch < 0) return fail(TREPB_ERR_INVALID, "batch must be >= 0");
    const RtSys& ps = s->P.proto;
    const size_t B = (size_t)batch, nq = ps.nd + ps.nk;
    CU(cudaSetDevice(s->device));
    Stager st(s);
    const double* dq1 = st.in(q1, B * nq); const double* dq2 = st.in(q2, B * nq); const double* dp1 = st.in(p1, B * ps.nd);
    const double* du = st.in(u1, B * ps.nu); const double* dl = st.in(lambda1, B * ps.nc);
    double* df = st.out(f, B * (ps.nd + ps.nc));
    const trepb_varied* dv = st.varied(v, B);
    if (st.err) return st.err;
    int rc = calc_f_dev(s, batch, t1, t2, dq1, dq2, dp1, du, dl, df, dv, nullptr);
    if (rc) return rc;
    return st.finish();
}

int trepb_calc_f_batch(trepb_system* s, int64_t batch, double t1, double t2, const double* q1, const double* q2,
                       const double* p1, const double* u1, const double* lambda1, double* f) {
    TREPB_NVTX("trepb_calc_f_batch");
    return calc_f_host(s, batch, t1, t2, q1, q2, p1, u1, lambda1, f, nullptr);
}

int trepb_calc_f_varied_batch(trepb_system* s, int64_t batch, double t1, double t2, const double* q1,
                              const double* q2, const double* p1, const double* u1, const double* lambda1, double* f,
                              const trepb_varied* v) {
    TREPB_NVTX("trepb_calc_f_varied_batch");
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    return calc_f_host(s, batch, t1, t2, q1, q2, p1, u1, lambda1, f, v);
}

static int discrete_fm2_host(trepb_system* s, int64_t batch, double t1, double t2, const double* q1,
                             const double* q2, const double* u1, double* fm2, const trepb_varied* v) {
    if (!s) return fail(TREPB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> hlk(s->mu_host);
    if (batch < 0) return fail(TREPB_ERR_INVALID, "batch must be >= 0");
    const RtSys& ps = s->P.proto;
    const size_t B = (size_t)batch, nq = ps.nd + ps.nk;
    CU(cudaSetDevice(s->device));
    Stager st(s);
    const double* dq1 = st.in(q1, B * nq); const double* dq2 = st.in(q2, B * nq);
    const double* du = st.in(u1, B * ps.nu);
    double* df = st.out(fm2, B * ps.nd);
    const trepb_varied* dv = st.varied(v, B);
    if (st.err) return st.err;
    int rc = discrete_fm2_dev(s, batch, t1, t2, dq1, dq2, du, df, dv, nullptr);
    if (rc) return rc;
    return st.finish();
}

int trepb_discrete_fm2_batch(trepb_system* s, int64_t batch, double t1, double t2, const double* q1,
                             const double* q2, const double* u1, double* fm2) {
    TREPB_NVTX("trepb_discrete_fm2_batch");
    return discrete_fm2_host(s, batch, t1, t2, q1, q2, u1, fm2, nullptr);
}

int trepb_discrete_fm2_varied_batch(trepb_system* s, int64_t batch, double t1, double t2, const double* q1,
                                    const double* q2, const double* u1, double* fm2, const trepb_varied* v) {
    TREPB_NVTX("trepb_discrete_fm2_varied_batch");
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    return discrete_fm2_host(s, batch, t1, t2, q1, q2, u1, fm2, v);
}

}  // extern "C"
namespace {
void stage_lin(Stager& st, const trepb_system* s, const trepb_lin_args* a, trepb_lin_args* d) {
    const RtSys& ps = s->P.proto;
    const size_t B = (size_t)a->batch, nq = ps.nd + ps.nk, nd = ps.nd, nu = ps.nu, nk = ps.nk, nc = ps.nc;
    const size_t nX = 2 * nq, nU = nu + nk;
    // state rows: [R][L] trajectories when traj_len is set (the caller's q2_guess then has the rows from its
    // start to the end of the q1 block only when it aliases q1; a separate q2_guess array must hold BS rows)
    const size_t BS = a->traj_len > 1 ? B / (size_t)(a->traj_len - 1) * (size_t)a->traj_len : B;
    *d = *a;
    d->t1 = st.in(a->t1, B); d->t2 = st.in(a->t2, B);
    d->q1 = st.in(a->q1, BS * nq); d->p1 = st.in(a->p1, BS * nd); d->u1 = st.in(a->u1, B * nu); d->k2 = st.in(a->k2, B * nk);
    if (a->traj_len > 1 && a->q2_guess == a->q1 + nq && nd == nq) d->q2_guess = d->q1 + nq;   // X[k+1] as the hint: no second copy
    else d->q2_guess = st.in(a->q2_guess, BS * nd);
    d->lambda_guess = st.in(a->lambda_guess, B * nc);
    d->q2 = st.out(a->q2, B * nq); d->p2 = st.out(a->p2, B * nd); d->lambda1 = st.out(a->lambda1, B * nc);
    d->iters = st.out(a->iters, B); d->status = st.out(a->status, B);
    d->A = st.out(a->A, B * nX * nX); d->B = st.out(a->B, B * nX * nU);
    d->q2_dq1 = st.out(a->q2_dq1, B * nq * nd); d->q2_dp1 = st.out(a->q2_dp1, B * nd * nd);
    d->q2_du1 = st.out(a->q2_du1, B * nu * nd); d->q2_dk2 = st.out(a->q2_dk2, B * nk * nd);
    d->p2_dq1 = st.out(a->p2_dq1, B * nq * nd); d->p2_dp1 = st.out(a->p2_dp1, B * nd * nd);
    d->p2_du1 = st.out(a->p2_du1, B * nu * nd); d->p2_dk2 = st.out(a->p2_dk2, B * nk * nd);
    d->l1_dq1 = st.out(a->l1_dq1, B * nq * nc); d->l1_dp1 = st.out(a->l1_dp1, B * nd * nc);
    d->l1_du1 = st.out(a->l1_du1, B * nu * nc); d->l1_dk2 = st.out(a->l1_dk2, B * nk * nc);
}
}  // namespace
extern "C" {

static int d2_host(trepb_system* s, const trepb_d2_args* a, const trepb_varied* v) {
    if (!s || !a) return fail(TREPB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> hlk(s->mu_host);
    if (a->lin.batch < 0) return fail(TREPB_ERR_INVALID, "batch must be >= 0");
    const RtSys& ps = s->P.proto;
    const size_t B = (size_t)a->lin.batch, nq = ps.nd + ps.nk, nd = ps.nd, nu = ps.nu, nk = ps.nk, nc = ps.nc;
    CU(cudaSetDevice(s->device));
    Stager st(s);
    trepb_d2_args d = *a;
    stage_lin(st, s, &a->lin, &d.lin);
    const size_t cnt[4] = {nq, nd, nu, nk};
    static const int ka[10] = {0, 0, 0, 0, 1, 1, 1, 2, 2, 3}, kb[10] = {0, 1, 2, 3, 1, 2, 3, 2, 3, 3};
    for (int w = 0; w < 3; ++w)
        for (int kd = 0; kd < 10; ++kd)
            d.d2[10 * w + kd] = st.out(a->d2[10 * w + kd], B * cnt[ka[kd]] * cnt[kb[kd]] * (w == 2 ? nc : nd));
    {
        const size_t nX = 2 * nq, nU = nu + nk;
        d.z = st.in(a->z, B * nX);
        d.fdxdx = st.out(a->fdxdx, B * nX * nX);
        d.fdxdu = st.out(a->fdxdu, B * nX * nU);
        d.fdudu = st.out(a->fdudu, B * nU * nU);
    }
    const trepb_varied* dv = st.varied(v, B);   // one row per instance
    if (st.err) return st.err;
    int rc = d2_dev(s, &d, nullptr, dv);
    if (rc) return rc;
    return st.finish();
}

int trepb_deriv2_batch(trepb_system* s, const trepb_d2_args* a) {
    TREPB_NVTX("trepb_deriv2_batch");
    return d2_host(s, a, nullptr);
}

int trepb_deriv2_varied_batch(trepb_system* s, const trepb_d2_args* a, const trepb_varied* v) {
    TREPB_NVTX("trepb_deriv2_varied_batch");
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    return d2_host(s, a, v);
}

static int lin_host(trepb_system* s, const trepb_lin_args* a, const trepb_varied* v) {
    if (!s || !a) return fail(TREPB_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> hlk(s->mu_host);
    if (a->batch < 0) return fail(TREPB_ERR_INVALID, "batch must be >= 0");
    CU(cudaSetDevice(s->device));
    // a large plain batch (no trajectory rows): chunks alternating between two streams (Pipe)
    if (const int C_ = Pipe::chunks((size_t)a->batch); C_ > 1 && a->traj_len <= 1 && a->q1 && a->p1 && a->status) {
        const RtSys& ps = s->P.proto;
        const size_t nq = ps.nd + ps.nk, nd = ps.nd, nu = ps.nu, nk = ps.nk, nc = ps.nc, nX = 2 * nq, nU = nu + nk;
        constexpr bool kIn = Pipe::kIn, kOut = Pipe::kOut;
        return Pipe(s, (size_t)a->batch).run(*a, v, C_, [&](trepb_lin_args& x, auto&& f) {
            f(x.t1, 1, kIn); f(x.t2, 1, kIn); f(x.q1, nq, kIn); f(x.p1, nd, kIn); f(x.u1, nu, kIn); f(x.k2, nk, kIn);
            f(x.q2_guess, nd, kIn); f(x.lambda_guess, nc, kIn);
            f(x.q2, nq, kOut); f(x.p2, nd, kOut); f(x.lambda1, nc, kOut); f(x.iters, 1, kOut); f(x.status, 1, kOut);
            f(x.A, nX * nX, kOut); f(x.B, nX * nU, kOut);
            f(x.q2_dq1, nq * nd, kOut); f(x.q2_dp1, nd * nd, kOut); f(x.q2_du1, nu * nd, kOut); f(x.q2_dk2, nk * nd, kOut);
            f(x.p2_dq1, nq * nd, kOut); f(x.p2_dp1, nd * nd, kOut); f(x.p2_du1, nu * nd, kOut); f(x.p2_dk2, nk * nd, kOut);
            f(x.l1_dq1, nq * nc, kOut); f(x.l1_dp1, nd * nc, kOut); f(x.l1_du1, nu * nc, kOut); f(x.l1_dk2, nk * nc, kOut);
        }, [&](const trepb_lin_args* e, const trepb_varied* ev, cudaStream_t st) { return lin_dev(s, e, st, ev); });
    }
    Stager st(s);
    trepb_lin_args d;
    stage_lin(st, s, a, &d);
    // one row per instance, or per trajectory
    const trepb_varied* dv = st.varied(v, a->traj_len > 1 ? (size_t)a->batch / (size_t)(a->traj_len - 1) : (size_t)a->batch);
    if (st.err) return st.err;
    int rc = lin_dev(s, &d, nullptr, dv);
    if (rc) return rc;
    return st.finish();
}

int trepb_linearize_batch(trepb_system* s, const trepb_lin_args* a) {
    TREPB_NVTX("trepb_linearize_batch");
    return lin_host(s, a, nullptr);
}

int trepb_linearize_varied_batch(trepb_system* s, const trepb_lin_args* a, const trepb_varied* v) {
    TREPB_NVTX("trepb_linearize_varied_batch");
    if (!v) return fail(TREPB_ERR_INVALID, "null trepb_varied");
    return lin_host(s, a, v);
}

}  // extern "C"

// ---- FP64 roofline denominator ------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) dfma_kernel(double* out, int iters, double a, double b) {
    double x0 = threadIdx.x * 1e-3, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; ++i) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}
}  // namespace

extern "C" int trepb_measure_fp64_peak(int device, double* tflops) {
    if (!tflops) return fail(TREPB_ERR_INVALID, "null argument");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 15;
    double* out = nullptr;
    CU(cudaMalloc((void**)&out, (size_t)blocks * threads * sizeof(double)));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(e0, 0));
        dfma_kernel<<<blocks, threads>>>(out, iters, 0.999999, 1e-7);
        CU(cudaEventRecord(e1, 0));
        CU(cudaEventSynchronize(e1));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        const double fl = 2.0 * 8.0 * (double)iters * blocks * threads;
        const double tf = fl / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    *tflops = best;
    return TREPB_OK;
}

// ---- diagnostic: the device sin / cos routine of the kernels (trepb_math.cuh sincos_dev) ----------
namespace {
__global__ void sincos_kernel(const double* x, double* s, double* c, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) trepb::sincos_(x[i], s + i, c + i);
}
}  // namespace

extern "C" int trepb_sincos_batch(int device, int64_t n, const double* x, double* s, double* c) {
    TREPB_NVTX("trepb_sincos_batch");
    if (n < 0 || (n > 0 && (!x || !s || !c))) return fail(TREPB_ERR_INVALID, "null argument");
    if (n == 0) return TREPB_OK;
    CU(cudaSetDevice(device));
    double *dx = nullptr, *ds = nullptr, *dc = nullptr;
    int rc = TREPB_OK;
    cudaError_t e = cudaMalloc((void**)&dx, n * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc((void**)&ds, n * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc((void**)&dc, n * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(dx, x, n * sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        sincos_kernel<<<(unsigned)((n + 255) / 256), 256>>>(dx, ds, dc, n);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(s, ds, n * sizeof(double), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(c, dc, n * sizeof(double), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) rc = cuda_fail(e, "trepb_sincos_batch");
    cudaFree(dx); cudaFree(ds); cudaFree(dc);
    return rc;
}
