// TEST INFRASTRUCTURE: g++ build of the cooperative kernels' link-level condensation (trep_b200/csrc/trepb_coop_sys.h),
// so that its split into a plan and a numeric evaluation is pinned on a machine without a GPU.
#include "../trep_b200/csrc/trepb_coop_sys.h"

using namespace trepb;

extern "C" {

// coop_pack(d): the blob followed by grav[3].  Returns its length in bytes (-1: the cooperative path does not apply),
// writes up to cap bytes.
int cvc_blob(const trepb_sysdesc* d, char* out, int cap) {
    CoopPack C = coop_pack(d);
    if (!C.ok) return -1;
    std::vector<char> v(C.blob);
    const char* g = (const char*)C.proto.grav;
    v.insert(v.end(), g, g + 3 * sizeof(double));
    for (size_t i = 0; i < v.size() && (int)i < cap; ++i) out[i] = v[i];
    return (int)v.size();
}

// The plan of coop_pack(d) evaluated on the table-driven expansion of one row (trepb_varied.h, slots = 0), in the
// layout of cvc_blob.  -1: invalid entries, or the cooperative path does not apply.
int cvc_expand(const trepb_sysdesc* d, int n, const int32_t* table, const int32_t* index, const double* row, char* out,
               int cap) {
    PackedSys P;
    std::string err;
    if (!pack_system(d, &P, &err) || !varied_check(P, n, table, index, &err)) return -1;
    CoopPack C = coop_pack(d);
    if (!C.ok) return -1;
    VariedHost H;
    varied_map(P, n, table, index, false, &H);
    const VariedX x{H.host_view(), row};
    const CoopPlanView pl = C.plan.view(C.plan.ints.data());
    std::vector<double> fx((size_t)12 * C.plan.nf, -7.0);
    std::vector<char> v(C.blob);
    for (int L = 0; L < pl.nlev; ++L) coop_eval_level(pl, x, fx.data(), L, 0, 1);
    coop_eval_tables(pl, x, fx.data(), (double*)v.data(), 0, 1);
    double g[3];
    for (int k = 0; k < 3; ++k) g[k] = x(pl.xg + k);
    v.insert(v.end(), (const char*)g, (const char*)g + sizeof(g));
    for (size_t i = 0; i < v.size() && (int)i < cap; ++i) out[i] = v[i];
    return (int)v.size();
}

}  // extern "C"
