// Launch interface of the team-cooperative kernels (trepb_coop.cu, trepb_coop_kernels.cuh).
#pragma once
#include <cuda_runtime.h>
#include "trepb_kernels.cuh"
#include "trepb_coop_math.cuh"

namespace trepb {

namespace coopk {
// most instances (one warp each) a CTA of the solve-only kernels (step, project, p2 / f) holds: their workspace
// is smaller than the linearize kernel's (CoopLayout::make, solve_only), 12 x 18.0 KB for the marionette
constexpr int kSolveTeams = 12;
// most instances a CTA of the linearize kernel holds (255 registers per thread with one warp per instance)
constexpr int kLinTeams = 8;
// the same for the flavours that keep part of the first-derivative workspace in global memory (ExtDims)
constexpr int kExtLinTeams = 16;
constexpr int kExtSolveTeams = 16;
// teams per CTA of the wide instantiations (shapes with small workspaces): 16 warps at 128 registers for the
// compile-time-size flavours, kWideTeamsRt warps for the run-time-size one
constexpr int kWideTeamsCt = 16;
#ifndef TREPB_WIDE_RT
#define TREPB_WIDE_RT 24
#endif
constexpr int kWideTeamsRt = TREPB_WIDE_RT;
}  // namespace coopk

struct CoopLaunch {
    int grid, warps;        // CTAs, teams (= instances in flight) per CTA; a team is team_warps warps
    size_t smem;            // table blob + warps x workspace
    cudaStream_t stream;
    CoopSys sys;            // view whose base is the DEVICE copy of the blob
    int blob_bytes;
    CoopLayout lay;
    double* ext;            // external slabs, grid x warps x lay.xtotal doubles (linearize kernels of ext flavours), or null
};

// What a varied launch (TREPB_FLAG_COOP_VARIED) hands the cooperative kernels besides their usual parameters.  Every
// team of the persistent grid owns a slot of `scratch`: a copy of the blob whose numeric tables it re-evaluates from
// its instance's row (coop_eval_level / coop_eval_tables, trepb_coop_sys.h) whenever the row changes, followed by the
// frame poses of that evaluation.  The team's view of the system points at the slot instead of the shared-memory copy.
struct CoopVaried {
    VariedMap map;          // the table-driven layout (trepb_varied.h, slots = false)
    const double* values;   // [rows][map.n]
    CoopPlanView plan;      // device pointers
    double* scratch;        // [grid x teams][per_team]
    long per_team;          // doubles: blob (rounded up to an even count) + 12 x frames
};

// One set per size flavour: run-time sizes ("cooperative") or a CtDims instantiation that serves
// every system of that shape (e.g. "cooperative/puppet").
struct CoopKernelSet {
    const char* name;
    int specialized;
    int team_warps;         // warps that work on one instance (1: WarpTeam, 2: PairTeam)
    int max_teams;          // teams per CTA of the wide instantiations (0: none; then lin_teams / kSolveTeams bound)
    int lin_teams;          // teams per CTA the base linearize instantiation is built for
    int solve_teams;        // ... and the base step / project / p2 instantiations
    int ext;                // 1: the linearize kernel keeps blocks in an external slab (CoopLayout::make, ext)
    bool (*matches)(const CoopSys&);
    cudaError_t (*step)(const CoopLaunch&, const StepParams&);
    cudaError_t (*p2)(const CoopLaunch&, const P2Params&);
    cudaError_t (*lin)(const CoopLaunch&, const LinParams&, const AuxLayout&);
    cudaError_t (*proj)(const CoopLaunch&, const ProjParams&);
    cudaError_t (*info)(int which, KernelInfo*);   // 0 step, 1 p2, 2 lin, 3 project
    // per-instance parameters: the *_varied_kernel instantiations of the same flavour and width
    cudaError_t (*step_v)(const CoopLaunch&, const StepParams&, const CoopVaried&);
    cudaError_t (*p2_v)(const CoopLaunch&, const P2Params&, const CoopVaried&);
    cudaError_t (*lin_v)(const CoopLaunch&, const LinParams&, const AuxLayout&, const CoopVaried&);
    cudaError_t (*proj_v)(const CoopLaunch&, const ProjParams&, const CoopVaried&);
};

struct CoopRegistry {
    static constexpr int kMax = 32;
    const CoopKernelSet* sets[kMax];
    int n;
};
CoopRegistry& coop_registry();
// layout fingerprint of what a cooperative specialisation unit shares with the library (see kSpecAbi)
constexpr unsigned kCoopAbi = 0x20000u + (unsigned)(sizeof(CoopSys) * 131 + sizeof(CoopLayout) * 31 + sizeof(CoopLaunch) * 17 +
                                                    sizeof(CoopKernelSet) * 13 + sizeof(StepParams) * 7 + sizeof(LinParams) * 5 +
                                                    sizeof(ProjParams) * 3 + sizeof(P2Params) + sizeof(CoopVaried) * 11);
bool coop_register(const CoopKernelSet* ks, unsigned abi);
struct CoopRegistrar {
    explicit CoopRegistrar(const CoopKernelSet* ks) { coop_register(ks, kCoopAbi); }
};
const CoopKernelSet* coop_general_kernels();
const CoopKernelSet* coop_select(const CoopSys& s, bool allow_specialized, int team_warps = 0);

}  // namespace trepb
